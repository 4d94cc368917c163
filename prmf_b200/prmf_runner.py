"""Drop-in for the reference CLI `script/prmf_runner.py` (main, :870-1093): same flags, same input
formats (delimited matrix with optional header / row names, graphml pathways with a `name` node
attribute, whitespace-delimited nodelist), same outputs (U.csv, V.csv, obj.txt, init_pathways.txt,
test_error.csv), same stdout lines and exit codes (22/23 manifold flags, 24 no pathway node in the
nodelist, 25 no nodelist and no header).  The factorisation itself runs on the GPU through
`prmf_b200.nmf_pathway`.

Differences from the reference, all deliberate (SURVEY.md section 0):
  * `--normalize` is accepted (no-op); `--high-dimensional false` really is false;
  * when the data is transposed (`--high-dimensional`, :946-952) the sample names follow the transpose,
    so writing U.csv no longer fails with an index-length mismatch;
  * `--m-samples` limits the rows read (the reference assigns the wrong variable, :933-935).
"""
import argparse
import copy
import csv
import os
import random
import sys
from argparse import RawTextHelpFormatter

import numpy as np

from . import prmf_args
from .manifold_init import pathway_init
from .solver import nmf_pathway


# ---- helpers from prmf/__init__.py that the CLI needs ----------------------------------------------
def relabel_nodes(G, node_attribute):
    """Use <node_attribute> as the node identifier where a node has it (prmf/__init__.py:65-76)."""
    import networkx as nx
    if node_attribute is not None:
        mapping = {n: d[node_attribute] for n, d in G.nodes(data=True) if node_attribute in d}
        G = nx.relabel_nodes(G, mapping)
    return G


def parse_nodelist(fh):
    """Whitespace-delimited identifiers, index = position (prmf/__init__.py:247-257)."""
    rv = []
    for line in fh:
        rv.extend(line.rstrip().split())
    return rv


def embed_arr(all_col_names, some_col_names, arr):
    """Place the columns of <arr> into a wider zero array ordered by <all_col_names>
    (prmf/__init__.py:331-352; one fancy-indexed assignment instead of an m x n Python loop)."""
    m, n = arr.shape
    if len(some_col_names) != n:
        raise ValueError("some_col_names != #columns of arr: {} != {}".format(len(some_col_names), n))
    index = {name: i for i, name in enumerate(all_col_names)}
    cols = np.fromiter((index[name] for name in some_col_names), dtype=np.int64, count=n)
    rv = np.zeros((m, len(all_col_names)))
    rv[:, cols] = arr
    return rv


def measure_cv_performance(gene_by_latent_train, data_test):
    """Per held-out sample: ||x - V u*|| / ||x|| with u* = argmin_{u>=0} (prmf/__init__.py:768-798), one batched
    solve on the GPU (prmf_b200.cv) instead of a scipy.optimize.nnls call per sample."""
    from .cv import measure_cv_performance as gpu_cv
    return gpu_cv(np.asarray(gene_by_latent_train), np.asarray(data_test))


def check_header(fpath, delim):
    """True when the first line has a non-numeric field (:794-808)."""
    with open(fpath, "r") as fh:
        for line in fh:
            for word in line.rstrip().split(delim):
                try:
                    float(word)
                except ValueError:
                    return True
            break
    return False


def check_row_names(fpath, delim, has_header):
    """True when the first field of the first data line is non-numeric (:810-831)."""
    target = 2 if has_header else 1
    data_line = None
    with open(fpath, "r") as fh:
        for i, line in enumerate(fh, start=1):
            data_line = line.rstrip()
            if i >= target:
                break
    try:
        float(data_line.split(delim)[0])
    except ValueError:
        return True
    return False


def parse_pathways(manifold_fps, node_attribute="name"):
    """graphml -> undirected graphs keyed by the `name` attribute (:833-868)."""
    import networkx as nx
    pairs = []
    for fp in manifold_fps:
        G = nx.read_graphml(fp).to_undirected()
        pairs.append((relabel_nodes(G, node_attribute), fp))
    return pairs


DESCRIPTION = """
Pathway-regularised matrix factorisation on NVIDIA B200 GPUs: X (samples x genes) is approximated by U V^T with U >= 0,
and every column of V is pulled towards the pathway graph it ends up assigned to.

  objective = ||X - U V^T||_F  +  gamma * sum_k vhat_k^T Lhat_{p(k)} vhat_k  +  delta * sum_k sum_{i in p(k)} 1 / (vhat_ik + 1)
              +  ||U||_F^2

  p(k)   pathway assigned to factor k (sampled among the remaining candidates, pruned every 10 steps, matched at the end)
  Lhat   normalised Laplacian of that pathway's graph, vhat_k = V[:,k] / ||V[:,k]||
  U: samples x k     V: genes x k

Same flags, inputs (--data, --manifolds *.graphml, --nodelist) and outputs (U.csv, V.csv, obj.txt) as prmf_runner.py of
gitter-lab/prmf; the multiplicative updates follow Cai et al. 2008 (NMF on manifold).
"""


def main(argv=None):
    import pandas as pd
    parser = argparse.ArgumentParser(description=DESCRIPTION, formatter_class=RawTextHelpFormatter)
    prmf_args.add_prmf_arguments(parser)
    args = parser.parse_args(argv)

    tradeoff = None if args.tradeoff == -1 else args.tradeoff                    # :894-897

    if args.manifolds is None and args.manifolds_file is None:                   # :901-914
        sys.stderr.write("Exactly one of --manifolds or --manifolds-file is required.\n")
        sys.exit(22)
    elif args.manifolds is None:
        with open(args.manifolds_file, "r") as fh:
            manifold_fps = [line.rstrip() for line in fh]
    elif args.manifolds_file is None:
        manifold_fps = args.manifolds
    else:
        sys.stderr.write("Exactly one of --manifolds or --manifolds-file is required.\n")
        sys.exit(23)
    G_fp_pairs = parse_pathways(manifold_fps)                                    # :915 (always by "name")
    fp_to_G = {fp: G for G, fp in G_fp_pairs}
    Gs = [G for G, _ in G_fp_pairs]

    if args.seed is not None:                                                    # :923-926
        seed = int(args.seed)
        np.random.seed(seed)
        random.seed(seed)

    has_header = check_header(args.data, args.delimiter)                         # :928-929
    has_row_names = check_row_names(args.data, args.delimiter, has_header)
    X = pd.read_csv(args.data, sep=args.delimiter, header="infer" if has_header else None,
                    nrows=None, index_col=0 if has_row_names else None)          # :942 (--m-samples never reaches it, :933-935)
    m, n = X.shape                                                               # :946-952, only when the flag is given
    if args.high_dimensional is not None and ((args.high_dimensional and m > n) or (not args.high_dimensional and m < n)):
        X = X.transpose()
    samples = list(X.index)

    if args.nodelist is not None:                                                # :957-975
        with open(args.nodelist) as fh:
            nodelist = parse_nodelist(fh)
        X = X.to_numpy()
    elif has_header:
        nodelist = list(X.columns)
        seen = set(nodelist)
        for G in Gs:
            for node in G:
                if node not in seen:
                    nodelist.append(node)
                    seen.add(node)
        X = embed_arr(nodelist, list(X.columns), X.to_numpy())
    else:
        sys.stderr.write("--nodelist is not provided and there is no header in <--data>\n")
        sys.exit(25)

    nodelist_set = set(nodelist)                                                 # :977-996
    fracs = []
    for G in Gs:
        count = sum(1 for node in G.nodes() if node in nodelist_set)
        fracs.append(count / G.order())
    if not any(f > 0 for f in fracs):
        sys.stderr.write("Invalid manifolds. Check that the node identifiers of the manifolds are present in the nodelist. Try setting --node-attribute if the node identifier is in a graphml attribute rather than the XML node attribute 'id'\n")
        sys.exit(24)
    sys.stdout.write("Printing manifold node representation in nodelist:\n")
    for (G, fp), frac in zip(G_fp_pairs, fracs):
        sys.stdout.write("{}: {:2.1f}%\n".format(fp, frac * 100))

    os.makedirs(args.outdir, exist_ok=True)
    U_fp = os.path.join(args.outdir, "U.csv")
    V_fp = os.path.join(args.outdir, "V.csv")
    obj_fp = os.path.join(args.outdir, "obj.txt")

    X_test = None                                                                # :1004-1013
    if args.cross_validation is not None:
        from sklearn.model_selection import KFold
        kf = KFold(n_splits=round(1 / args.cross_validation))
        for train_index, test_index in kf.split(X):
            X_test = X[test_index]
            X = X[train_index]
            samples = [samples[i] for i in train_index]
            break

    if not args.no_normalize:                                                    # :1019-1020
        # sklearn.preprocessing.quantile_transform(X) on the GPU; the result stays on the device for nmf_pathway
        from .preprocess import quantile_transform
        X = quantile_transform(np.asarray(X, dtype=np.float64), return_device=True)

    U_init = V_init = None                                                       # :1023-1064
    if args.manifolds_init is not None:
        Gs_init = [fp_to_G[fp] for fp in args.manifolds_init]
        if len(args.manifolds_init) < args.k_latent:
            non_init = list(set(manifold_fps) - set(args.manifolds_init))
            chosen = random.sample(non_init, args.k_latent - len(args.manifolds_init))
            init_fps = copy.copy(args.manifolds_init)
            for fp in chosen:
                Gs_init.append(fp_to_G[fp])
                init_fps.append(fp)
        elif len(args.manifolds_init) == args.k_latent:
            init_fps = args.manifolds_init
        else:
            inds = np.random.choice(len(Gs_init), args.k_latent)
            init_fps = [args.manifolds_init[i] for i in inds]
            Gs_init = [Gs_init[i] for i in inds]
        # pathway_to_vec -> nmf_init_u -> nmf_init_v for every init pathway (:272-334, :1023-1064), batched on the GPU
        # against X where it already lives
        U_init, V_init = pathway_init(X, Gs_init, nodelist)
        sys.stdout.write("Using the following manifolds for initialization:\n{}\n".format("\n".join(init_fps)))
        with open(os.path.join(args.outdir, "init_pathways.txt"), "w") as fh:
            fh.write("\n".join(init_fps))

    # :1067 -- like the reference only gamma, tradeoff, k_latent, U_init, V_init and verbose are forwarded
    U, V, obj_data = nmf_pathway(X, Gs, nodelist=nodelist, gamma=args.gamma, tradeoff=tradeoff,
                                 k_latent=args.k_latent, U_init=U_init, V_init=V_init, verbose=args.verbose)
    cols = ["LV{}".format(i) for i in range(args.k_latent)]
    pd.DataFrame(U, index=samples, columns=cols).to_csv(U_fp, sep=",", index=has_row_names, quoting=csv.QUOTE_NONNUMERIC)
    V_df = pd.DataFrame(V, index=nodelist, columns=cols)
    V_df.to_csv(V_fp, sep=",", index=True, quoting=csv.QUOTE_NONNUMERIC)

    latent_to_pathway_data = obj_data.pop("latent_to_pathway_data", {})

    def write_obj():                                                             # :1081-1093
        with open(obj_fp, "w") as fh:
            for key, val in obj_data.items():
                fh.write("{} = {:0.5f}\n".format(key, val))
            for k in sorted(latent_to_pathway_data.keys()):
                lapl_ind = latent_to_pathway_data[k][0][0]
                fh.write("{} -> {}\n".format(k, G_fp_pairs[lapl_ind][1]))

    if args.cross_validation is not None:                                        # :1074-1079
        write_obj()              # a failure of the hold-out scoring must not lose the objective of a finished run
        errs = measure_cv_performance(V_df, X_test)
        np.savetxt(os.path.join(args.outdir, "test_error.csv"), errs, delimiter=",")
        obj_data["average_normalized_test_error"] = np.mean(errs)
    write_obj()


if __name__ == "__main__":
    main()
