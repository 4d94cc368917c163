"""Inputs shared by make_golden.py and the tests (no reference import)."""
import os


def side_by_side_instance(seed):
    """The instances tests/test_oracle_golden.py::test_oracle_vs_live_reference runs (seed 1 has weighted edges)."""
    from prmf_b200 import synth
    return synth.small_instance(m=30, n=150, k_true=3, n_pathways=14, pathway_size=16, seed=20 + seed,
                                weighted=bool(seed))


def write_cli_inputs(outdir, X, nodelist, Gs, header=False):
    """data.tsv (+ header variant), nodelist.txt and graph{k}.graphml as test_inferred_nodelist_1.py writes
    them (:27-45): integer node ids with the gene symbol in the `name` attribute."""
    import networkx as nx
    import pandas as pd
    os.makedirs(outdir, exist_ok=True)
    df = pd.DataFrame(X, index=[str(i) for i in range(X.shape[0])], columns=nodelist)
    df.to_csv(os.path.join(outdir, "data.tsv"), sep="\t", header=False, index=False)
    df.to_csv(os.path.join(outdir, "data_header.tsv"), sep="\t", header=nodelist, index=False)
    with open(os.path.join(outdir, "nodelist.txt"), "w") as fh:
        fh.write("\n".join(nodelist))
    fps = []
    for k, G in enumerate(Gs):
        H = nx.Graph()
        ids = {g: i for i, g in enumerate(G.nodes())}
        for g, i in ids.items():
            H.add_node(i, name=g)
        for a, b in G.edges():
            H.add_edge(ids[a], ids[b])
        fp = os.path.join(outdir, "graph%d.graphml" % k)
        nx.write_graphml(H, fp)
        fps.append(fp)
    return fps


