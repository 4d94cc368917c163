"""Developer tool: wall time of the pathway-seeded initialisation (`--manifolds-init`, prmf_b200.pathway_init) at the
recount2 shape (config 2: 37 032 x 6 750, synth.recount2_shape) with 10 seeded pathways, next to the host scipy path
of the reference (tests/init_reference.py) for the first --host-factors factors of the same instance, in one run.

    python tools/init_timing.py --host-factors 1 --out profiles/init_timing_c2.json

GPU times: a host clock around the whole pathway_init call, which ends in a device synchronise (the results are on the
host), with X already on the device and with X in host memory (the upload included).  One untimed call first."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def device_env(dev):
    import torch
    env = {"device": torch.cuda.get_device_name(dev)}
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(dev), "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        env["power_limit"], env["max_sm_clock"] = [s.strip() for s in out.split(",")]
    except Exception as exc:                                       # reported, not guessed
        env["power_limit"] = "unavailable: %s" % exc
    return env


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--host-factors", type=int, default=1, help="factors solved by the host scipy path (0: none)")
    ap.add_argument("--reps", type=int, default=3, help="timed GPU calls per variant")
    ap.add_argument("--pathways", type=int, default=10)
    ap.add_argument("--m", type=int, default=37032)
    ap.add_argument("--n", type=int, default=6750)
    ap.add_argument("--out", default=None, help="also write the JSON result here")
    a = ap.parse_args()

    import torch
    from prmf_b200 import pathway_init, synth
    import init_reference as R

    if not torch.cuda.is_available():
        raise SystemExit("init_timing needs a CUDA device")
    dev = torch.cuda.current_device()
    res = {"instance": {"generator": "synth.recount2_shape", "m": a.m, "n": a.n, "pathways": a.pathways, "seed": 0}}
    res["env"] = device_env(dev)
    X, nodelist, Gs = synth.recount2_shape(m=a.m, n=a.n, n_pathways=a.pathways)
    res["instance"]["pathway_sizes"] = [G.number_of_nodes() for G in Gs]
    Xd = torch.from_numpy(X).to("cuda")
    torch.cuda.synchronize()

    stats = {}
    U, V = pathway_init(Xd, Gs, nodelist, stats=stats)             # untimed: module load, allocations into the pool
    res["lh_iterations"] = stats
    for label, src in (("x_on_device", Xd), ("x_from_host", X)):
        times = []
        for _ in range(a.reps):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            U2, V2 = pathway_init(src, Gs, nodelist)
            torch.cuda.synchronize()
            times.append(time.perf_counter() - t0)
            assert np.array_equal(U, U2) and np.array_equal(V, V2), "repeated init differs"
        res["gpu_seconds_" + label] = times
    res["gpu_seconds_whole_init_k%d" % a.pathways] = min(res["gpu_seconds_x_on_device"])

    host = []
    for c in range(min(a.host_factors, a.pathways)):
        t0 = time.perf_counter()
        v, on = R.pathway_to_vec(X, Gs[c], nodelist)
        t1 = time.perf_counter()
        u, _ = R.nmf_init_u(X, v)
        t2 = time.perf_counter()
        vn, _ = R.nmf_init_v(X, u)
        t3 = time.perf_counter()
        vn[on] = v[on]
        u, vn = u.ravel(), vn.ravel()
        host.append({
            "factor": c,
            "seconds_pathway_to_vec": t1 - t0, "seconds_nnls_Xt_v": t2 - t1, "seconds_nnls_X_u": t3 - t2,
            "seconds_total": t3 - t0,
            "nonzeros_u": int((u > 0).sum()), "nonzeros_v": int((vn > 0).sum() - on.sum()),
            "support_u_identical": bool(np.array_equal(u > 0, U[:, c] > 0)),
            "support_v_identical": bool(np.array_equal(vn > 0, V[:, c] > 0)),
            "max_rel_diff_u": float(np.abs(u - U[:, c]).max() / np.abs(u).max()),
            "max_rel_diff_v": float(np.abs(vn - V[:, c]).max() / np.abs(vn).max()),
        })
    res["host_scipy"] = host
    if host:
        res["host_seconds_per_factor"] = float(np.mean([h["seconds_total"] for h in host]))
    line = json.dumps(res, indent=1)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
