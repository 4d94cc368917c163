"""Host restatement of the reference's pathway-seeded initialisation (script/prmf_runner.py:272-334 and the loop at
:1023-1064), the checker for prmf_b200.manifold_init.  Test infrastructure: nothing under prmf_b200/ imports it."""
import numpy as np


def pathway_to_vec(X, G, nodelist, rel_weight=5):
    n_genes = len(nodelist)
    v = np.zeros((n_genes,))
    index = {node: i for i, node in enumerate(nodelist)}
    for node in G.nodes():
        v[index[node]] = 1
    on = (v == 1)
    off = np.invert(on)
    v[off] = np.mean(X.transpose()[off], axis=1)
    v[on] = (np.sum(v[off]) * rel_weight) / np.sum(on)
    v = v.reshape((n_genes, 1))
    return v / np.linalg.norm(v), on


def nmf_init_u(X, v):
    import scipy.optimize
    u, residual = scipy.optimize.nnls(X.transpose(), v.flatten())
    return (u / np.linalg.norm(u) ** 2).reshape((X.shape[0], 1)), residual


def nmf_init_v(X, u):
    import scipy.optimize
    v, residual = scipy.optimize.nnls(X, u.flatten())
    return (v / np.linalg.norm(v) ** 2).reshape(X.shape[1], 1), residual


def pathway_init(X, Gs_init, nodelist):
    """The CLI's per-factor loop (:1023-1064): (U_init, V_init) with one column per init pathway."""
    us, vs = [], []
    for G in Gs_init:
        v, on = pathway_to_vec(X, G, nodelist)
        signal = v[on]
        u, _ = nmf_init_u(X, v)
        v_new, _ = nmf_init_v(X, u)
        v_new[on] = signal
        vs.append(v_new)
        us.append(u)
    return np.concatenate(us, axis=1), np.concatenate(vs, axis=1)
