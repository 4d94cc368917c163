"""Developer tool: the fp32 storage mode (x_dtype="f32") against the fp64 mode at BASELINE configs 2 and 4, in one process.

    python tools/f32_timing.py --out-dir profiles

Both handles hold the same matrix: bench.py's synthetic X rounded to fp32 (float32 for the f32 handle, its exact fp64
widening for the fp64 handle), the same pathways and the same U0 / V0.  The two modes run alternately, --rounds times:
each round times --steps outer iterations of each mode with the loop bench.py times (sample, set_active, step_async,
block_end with the score tables and the speculative next pass, restrict on the host), a host clock around work that
ends in a device synchronise, then the same outer iterations again in profiling mode for the per-phase device times
(set_profiling / kernel_times; with the fused tails at k <= 10 the "xv" and "xtu" phases include the U and V updates).
The warm-up iterations start both modes from the same state and RNG seed; their objective rows must be bitwise equal.
The device name and power limit are read in the same run.  Writes f32_timing_c2.json and f32_timing_c4.json."""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

MODES = ("f64", "f32")


def run_config(cfg, a, device_env):
    import torch
    import bench
    from prmf_b200 import CudaEngine
    from prmf_b200.solver import init_latent_to_pathway_data, restrict_from_tables, sample_active

    ba = argparse.Namespace(**bench.CONFIGS[cfg])
    m, n, k = ba.m, ba.n, ba.k
    Gs, nodelist, packed = bench.make_pathways(ba)
    X32 = bench.host_rows(0, m, n, np.float64).astype(np.float32)
    U0, V0 = bench.initial_UV(ba)
    engines = {}
    for mode in MODES:
        eng = CudaEngine(m, m, n, k, x_dtype=mode)
        eng.set_X(X32 if mode == "f32" else X32.astype(np.float64))
        eng.set_pathways(packed)
        engines[mode] = eng
    normX = float(np.sqrt(engines["f64"].normX_sq))
    assert engines["f32"].normX_sq == engines["f64"].normX_sq
    gamma, delta = normX / k, 10 / normX
    cands = init_latent_to_pathway_data(k, packed.P)

    def outer(eng):
        eng.set_active(sample_active(cands, k))
        eng.step_async(bench.MODULUS, gamma, delta)
        parts, _, _, (mass, qn, _) = eng.block_end(bench.MODULUS, want_scores=True, prefetch=True)
        restrict_from_tables(mass, qn, cands)
        return parts

    warm = {}
    for mode, eng in engines.items():
        eng.set_UV(U0, V0)
        np.random.seed(1)
        warm[mode] = np.concatenate([outer(eng) for _ in range(a.warmup)])
    torch.cuda.synchronize()
    res = {"config": cfg, "m": m, "n": n, "k": k, "pathways": ba.pathways, "steps": a.steps, "rounds": a.rounds,
           "warmup": a.warmup, "env": device_env, "X": "bench.py host_rows (seed %d) rounded to fp32" % bench.X_SEED,
           "warmup_objective_rows_bitwise_equal": bool(np.array_equal(warm["f32"], warm["f64"])),
           "modes": {mode: {"outer_it_per_s": [], "xv_ms": [], "xtu_ms": []} for mode in MODES}}
    for _ in range(a.rounds):
        for mode, eng in engines.items():
            np.random.seed(2)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(a.steps):
                outer(eng)
            torch.cuda.synchronize()
            res["modes"][mode]["outer_it_per_s"].append(a.steps / (time.perf_counter() - t0))
            eng.kernel_times(reset=True)
            eng.set_profiling(True)
            for _ in range(a.steps):
                outer(eng)
            eng.set_profiling(False)
            kt = eng.kernel_times(reset=True)
            for phase in ("xv", "xtu"):
                ms, cnt = kt[phase]
                res["modes"][mode][phase + "_ms"].append(ms / max(1, cnt))
    for mode in MODES:
        r = res["modes"][mode]
        r["median"] = {key: float(np.median(r[key])) for key in ("outer_it_per_s", "xv_ms", "xtu_ms")}
    # bytes of X one pass reads, and its DFMA count (2 flop per multiply-add)
    res["per_pass"] = {"bytes_f64": 8 * m * n, "bytes_f32": 4 * m * n, "flop": 2 * m * n * k}
    for eng in engines.values():
        eng.close()
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--configs", default="2,4")
    ap.add_argument("--steps", type=int, default=20, help="outer iterations per timed window")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3, help="alternations of the two modes")
    ap.add_argument("--out-dir", default=None, help="write f32_timing_c<config>.json here")
    a = ap.parse_args()
    import torch
    from init_timing import device_env
    if not torch.cuda.is_available():
        raise SystemExit("f32_timing needs a CUDA device")
    env = device_env(torch.cuda.current_device())
    for cfg in (int(c) for c in a.configs.split(",")):
        res = run_config(cfg, a, env)
        print(json.dumps({"config": cfg, "env": env, "equal": res["warmup_objective_rows_bitwise_equal"],
                          **{mode: res["modes"][mode]["median"] for mode in MODES}}), flush=True)
        if a.out_dir:
            os.makedirs(a.out_dir, exist_ok=True)
            with open(os.path.join(a.out_dir, "f32_timing_c%d.json" % cfg), "w") as fh:
                json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
