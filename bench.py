#!/usr/bin/env python
"""PRMF hot-path benchmark (contract: see the task statement / DESIGN.md "Measurement").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config 2|4|5] [--dump-outputs DIR]
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...

One *step* = one outer iteration of `nmf_pathway` (reference script/prmf_runner.py:715-774) on the
recount2-shape synthetic instance (BASELINE.json configs[1]: 37 032 samples x 6 750 genes, k = 10,
300 KEGG-size random pathways): k multinomial draws of the active pathways, `modulus` = 10 inner
multiplicative updates with their objectives, and one `restrict` over the full candidate table.
`value` is outer iterations per second with X resident in HBM; `e2e` is the same step driven with
host buffers (X, U, V uploaded from pinned memory and U, V, objective read back every step).
With N > 1 the rows of X and U are sharded over the ranks (strong scaling: the SAME global instance for
every N; one sum over ranks of [X^T U | U^T U] per inner step).

Every line also carries a `parity` block: two inner steps from fixed U0 / V0 and one `restrict`, computed by
the GPU path in this run and compared on rank 0 with the CPU reference on the same full-shape arrays
(U, V, the five objective parts, the surviving candidates), plus digests that must agree across ranks and
across N.  `--impl reference` times the reference's own CPU implementation (the unmodified
`prmf_runner.py` functions from `baseline/_ref` when that install travelled with the repo, else the oracle
port) on all host cores.

`--dump-outputs DIR` writes what the last timed step computed (objective parts, U, V, score tables, the
candidates `restrict` kept, in order) as float64 .npy files; the inputs depend only on the arguments, so two
builds can be compared output for output.
"""
import os
import sys

# torch.distributed.run exports OMP_NUM_THREADS=1 to every rank; the CPU legs (the reference arm, the parity
# check and the cpu_baseline) must use all host cores, and BLAS reads these variables when numpy loads
if "--impl" in sys.argv and "reference" in sys.argv or os.environ.get("RANK", "0") == "0":
    for _v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[_v] = str(os.cpu_count() or 1)

import argparse
import contextlib
import hashlib
import io
import json
import subprocess
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

MODULUS = 10
CONFIGS = {          # BASELINE.json configs[1] / [3] / [4]
    2: dict(m=37032, n=6750, k=10, pathways=300, x_dtype="f64"),
    4: dict(m=37032, n=6750, k=64, pathways=2000, x_dtype="f64"),
    5: dict(m=1000000, n=20000, k=128, pathways=2000, x_dtype="tf32"),
}
METRIC = "prmf_outer_iterations_per_sec"
UNIT = "outer_it/s"
X_SEED = 1234
X_BLOCK_ROWS = 4096
FP64_DFMA_PEAK_TFLOPS = 33.0      # measured with tools/fp64_microbench.cu on B200 (DESIGN.md section 3)
REF_SCRIPT = os.path.join(ROOT, "baseline", "_ref", "bin", "prmf_runner.py")


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=sorted(CONFIGS),
                    help="BASELINE.json configuration: 2 (headline), 4 (k=64, 2000 pathways), 5 (1M x 20k, k=128, tf32)")
    ap.add_argument("--m", type=int, default=None)
    ap.add_argument("--n", type=int, default=None)
    ap.add_argument("--k", type=int, default=None)
    ap.add_argument("--pathways", type=int, default=None)
    ap.add_argument("--x-dtype", default=None, choices=["f64", "tf32"],
                    help="f64: parity mode (default, the headline); tf32: opt-in tensor-core X streams (X stored fp32)")
    ap.add_argument("--x-gen", default=None, choices=["host", "device"],
                    help="where the synthetic X is drawn (default: host below 2^31 elements, else device)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-converge", action="store_true")
    ap.add_argument("--cpu-inner-steps", type=int, default=2)
    ap.add_argument("--ref-budget-s", type=float, default=150.0,
                    help="--impl reference: wall-clock budget that sizes the bounded sample of each step")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (float64, "
                         "at most 64 MB; U as a fixed, seeded row sample when it does not fit)")
    a = ap.parse_args()
    if a.steps < 1 or a.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")
    for key, val in CONFIGS[a.config].items():
        if getattr(a, key) is None:
            setattr(a, key, val)
    if a.x_gen is None:
        a.x_gen = "host" if a.m * a.n < (1 << 31) else "device"
    return a


def workload_name(a):
    return "recount2-shape synthetic %dx%d %s, k=%d, %d random KEGG-size pathways" % (
        a.m, a.n, "fp64" if a.x_dtype == "f64" else "fp32 (tf32 tensor-core X streams)", a.k, a.pathways)


def config_dict(a):
    """The same dict in both arms (the driver compares them)."""
    return {"workload": workload_name(a), "baseline_config": a.config,
            "step": "1 outer iteration = k multinomial draws + 10 inner steps + scores/restrict over all candidates",
            "x": "iid U(0,1), PCG64 seed %d per %d-row block (the same global matrix for every N); %s" % (
                X_SEED, X_BLOCK_ROWS, "drawn on the host" if a.x_gen == "host" else "drawn on the device"),
            "l2": "inputs larger than L2 (every pass streams the rank's whole X block)"}


def make_pathways(a):
    from prmf_b200 import pack_pathways, synth
    rng = np.random.Generator(np.random.PCG64(0))
    Gs = synth.random_pathway_graphs(rng, a.n, a.pathways)
    nodelist = list(range(a.n))
    return Gs, nodelist, pack_pathways(Gs, nodelist)


# ------------------------------------------------------------------------------------------------
# the synthetic X: one PCG64 stream per block of X_BLOCK_ROWS global rows, so that any row range of the SAME
# global matrix can be drawn by any rank (strong scaling compares one instance across N)
# ------------------------------------------------------------------------------------------------
def host_rows(lo, hi, n, dtype=np.float64, out=None):
    X = out if out is not None else np.empty((hi - lo, n), dtype=dtype)
    b0 = lo // X_BLOCK_ROWS
    b1 = (hi + X_BLOCK_ROWS - 1) // X_BLOCK_ROWS if hi > lo else b0
    for b in range(b0, b1):
        r0, r1 = b * X_BLOCK_ROWS, (b + 1) * X_BLOCK_ROWS
        rng = np.random.Generator(np.random.PCG64([X_SEED, b]))
        s0, s1 = max(lo, r0), min(hi, r1)
        blk = rng.random((s1 - r0, n))[s0 - r0:]             # rows r0 .. s1 of the block, in stream order
        X[s0 - lo:s1 - lo] = blk
    return X


def device_rows(lo, hi, n, torch_dtype):
    """Device-drawn variant for instances that do not fit host memory (config 5): torch's Philox stream per block."""
    import torch
    X = torch.empty((hi - lo, n), dtype=torch_dtype, device="cuda")
    gen = torch.Generator(device="cuda")
    b0 = lo // X_BLOCK_ROWS
    b1 = (hi + X_BLOCK_ROWS - 1) // X_BLOCK_ROWS if hi > lo else b0
    for b in range(b0, b1):
        r0, r1 = b * X_BLOCK_ROWS, (b + 1) * X_BLOCK_ROWS
        gen.manual_seed(X_SEED * 1000003 + b)
        s0, s1 = max(lo, r0), min(hi, r1)
        blk = torch.rand((X_BLOCK_ROWS, n), dtype=torch_dtype, device="cuda", generator=gen)
        X[s0 - lo:s1 - lo] = blk[s0 - r0:s1 - r0]
        del blk
    return X


def initial_UV(a):
    """The reference's initialisation (:650-655) from the legacy global RNG, seed 1."""
    np.random.seed(1)
    U0 = 3 * (1 - np.random.rand(a.m, a.k))
    V0 = 3 * (1 - np.random.rand(a.n, a.k))
    return U0, V0


def plant_signal(X, Gs, lo, m_global, n_plant=10):
    """SURVEY 8d: a rank-1 bump on the genes of the first `n_plant` pathways so that the assignment is not
    degenerate (X: rows lo.. of the global matrix, modified in place)."""
    rng = np.random.Generator(np.random.PCG64(77))
    for p in range(min(n_plant, len(Gs))):
        genes = np.fromiter(Gs[p].nodes(), dtype=np.int64)
        u = rng.random(m_global) * 0.5
        X[:, genes] += u[lo:lo + X.shape[0], None].astype(X.dtype)
    return X


def digest(arr):
    return hashlib.sha256(np.ascontiguousarray(arr).tobytes()).hexdigest()[:16]


# ------------------------------------------------------------------------------------------------
# --dump-outputs: what the last timed step computed, so that two builds can be compared output for output
# ------------------------------------------------------------------------------------------------
DUMP_BYTES = 60 << 20             # below 64 MB with room for the .npy headers
DUMP_SEED = 4321


def dump_rows(m, k, other_bytes):
    """Global rows of U (m x k, float64) to write beside `other_bytes` of other outputs: None for all of them, else a
    sorted sample drawn from a fixed seed (the same rows for the same shape, whatever the number of ranks)."""
    budget = DUMP_BYTES - other_bytes
    row_bytes = 8 * k + 8                          # a row of U and its index in U_rows
    if budget < row_bytes:
        raise SystemExit("bench.py: --dump-outputs: V and the score tables alone exceed %d bytes" % DUMP_BYTES)
    if m * 8 * k <= budget:
        return None
    rng = np.random.Generator(np.random.PCG64(DUMP_SEED))
    return np.sort(rng.choice(m, size=budget // row_bytes, replace=False))


def restrict_arrays(surv, k, P):
    """`restrict`'s result {factor: [(pathway, score), ...]} as two k x P arrays: the 1-based position of each surviving
    candidate in its factor's list (0: dropped), and its score.  The order counts: the next multinomial draw picks
    from the list by position."""
    position, scores = np.zeros((k, P)), np.zeros((k, P))
    for kk, cands in surv.items():
        for i, (p, s) in enumerate(cands):
            position[kk, int(p)] = i + 1
            scores[kk, int(p)] = s
    return position, scores


def dump_outputs(a, ctx, eng, lo, hi, last, P):
    """The last timed outer iteration's outputs: the objective parts of its 10 inner steps, U and V after them, the
    score tables and the candidates `restrict` kept.  Every rank takes part (U is gathered); rank 0 writes."""
    parts, mass, qn, surv = last
    U_local, V = eng.get_UV()
    position, scores = restrict_arrays(surv, a.k, P)
    out = {"obj_parts": parts[:, :5], "V": V, "score_mass": mass, "score_quad_norm": qn,
           "restrict_position": position, "restrict_scores": scores}
    rows = dump_rows(a.m, a.k, sum(np.asarray(v).nbytes for v in out.values()))
    sel = np.arange(a.m) if rows is None else rows
    out["U"] = ctx.all_gather_rows(U_local[sel[(sel >= lo) & (sel < hi)] - lo], len(sel))
    if rows is not None:
        out["U_rows"] = rows.astype(np.float64)
    if ctx.rank == 0:
        os.makedirs(a.dump_outputs, exist_ok=True)
        for name, arr in out.items():
            np.save(os.path.join(a.dump_outputs, name + ".npy"), np.ascontiguousarray(arr, dtype=np.float64))


# ------------------------------------------------------------------------------------------------
# clocks (nvidia-smi sampled during the timed region)
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.path = None
        self.begin = 0

    def _lines(self):
        try:
            with open(self.path) as fh:
                return fh.readlines()
        except Exception:
            return []

    def mark_begin(self):
        """Samples before this point (set-up, warm-up) are not part of the timed region."""
        self.begin = len(self._lines())

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                 "-lms", "20"], stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, smax, reasons, power = [], [], set(), []
        try:
            lines = self._lines()
            lines = lines[self.begin:] if len(lines) > self.begin else lines[-3:]
            for line in lines:
                f = [x.strip() for x in line.split(",")]
                if len(f) < 9:
                    continue
                try:
                    sm.append(float(f[1])); smax.append(float(f[2])); power.append(float(f[3]))
                except ValueError:
                    continue
                for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(smax)), reasons=sorted(reasons),
                       samples=len(sm), power_w_max=float(max(power)))
        return out


# ------------------------------------------------------------------------------------------------
# the CPU side: the reference's own functions (baseline/_ref) or the oracle port
# ------------------------------------------------------------------------------------------------
def host_threads():
    try:
        from threadpoolctl import threadpool_info
        n = [p.get("num_threads", 1) for p in threadpool_info() if p.get("user_api") == "blas"]
        if n:
            return int(max(n))
    except Exception:
        pass
    return os.cpu_count() or 1


def use_all_cores():
    try:
        from threadpoolctl import threadpool_limits
        threadpool_limits(limits=os.cpu_count() or 1)
    except Exception:
        pass


class CpuReference:
    """The CPU implementation of the path, timed and used as the parity checker of `bench.py`.

    kind "reference": the UNMODIFIED functions `nmf_manifold_vec_update` (:374-451) and `restrict` (:129-194) of the
    reference's `prmf_runner.py` as pip-installed into `baseline/_ref` (git-ignored; travels to the GPU box), fed
    with the per-pathway n x n scipy matrices its `nmf_pathway` builds (:670-696) and its module-global table of
    normalised Laplacians.  kind "port": `oracle/prmf_oracle.py` when that install is absent."""

    def __init__(self, Gs, nodelist, k, force_port=False):
        from oracle import prmf_oracle as O
        self.O = O
        self.k = k
        t0 = time.perf_counter()
        self.tables = O.PathwayTables(Gs, nodelist)       # W, D, L, supports (as :678-690) + normalised Laplacians
        self.mod = None
        self.kind = "port"
        if os.path.isfile(REF_SCRIPT) and not force_port:
            try:
                self.mod = self._load_reference()
                self.kind = "reference"
            except Exception as exc:                       # pragma: no cover - depends on the box
                sys.stderr.write("bench.py: baseline/_ref present but not importable (%s); using the oracle port\n" % exc)
        self.Ws, self.Ds, self.Ls = self.tables.Ws, self.tables.Ds, self.tables.Ls
        if self.mod is not None:
            import scipy.sparse as sp
            n = len(nodelist)
            # D and L in the storage formats the reference's nmf_pathway builds them in (:680-683): D is a DOK matrix
            self.Ds = [sp.dok_matrix(sp.dia_matrix((W.sum(axis=0), np.array([0])), shape=(n, n))) for W in self.Ws]
            self.Ls = [D - W for D, W in zip(self.Ds, self.Ws)]
            self.mod.PATHWAY_TO_SUPPORT = dict(enumerate(self.tables.supports))                          # :691
            self.mod.LAPLACIANS = self.Ls
            self.mod.NORMALIZED_LAPLACIANS = [self.mod.normalize_laplacian(L, s)
                                              for L, s in zip(self.Ls, self.tables.supports)]           # :693-696
        self.t_tables = time.perf_counter() - t0

    @staticmethod
    def _load_reference():
        import importlib.util
        if not hasattr(np, "Inf"):
            np.Inf = np.inf                                # the reference predates NumPy 2 (:713)
        sys.dont_write_bytecode = True
        ref_site = os.path.join(ROOT, "baseline", "_ref")
        if ref_site not in sys.path:
            sys.path.insert(0, ref_site)
        spec = importlib.util.spec_from_file_location("prmf_runner_reference", REF_SCRIPT)
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        return mod

    def inner_steps(self, X, U, V, active, n_steps, gamma, delta, norm_X):
        """`n_steps` inner steps; returns U, V and the objective parts of every step [n_steps, 5]."""
        if self.mod is None:
            log = []
            U, V, _, _, _ = self.O.update_block(X, U, V, self.tables, active, n_steps, gamma, delta, None, log)
            return U, V, np.array([[d[key] for key in ("recon", "manifold", "ignore", "fro", "obj")] for d in log])
        k_to_W = {kk: self.Ws[p] for kk, p in enumerate(active)}                 # map_k_to_lapls (:260-270)
        k_to_D = {kk: self.Ds[p] for kk, p in enumerate(active)}
        k_to_L = {kk: self.Ls[p] for kk, p in enumerate(active)}
        k_to_feat = {kk: self.tables.supports[p] for kk, p in enumerate(active)}
        parts = []
        for s in range(n_steps):          # one call per step to see every step's objective parts (:446-447)
            with contextlib.redirect_stdout(io.StringIO()):
                U, V, od = self.mod.nmf_manifold_vec_update(X, U, V, k_to_W, k_to_D, k_to_L, k_to_feat, n_steps=1,
                                                            gamma=gamma, delta=delta, i=s, verbose=False, norm_X=norm_X)
            parts.append([od[key] for key in ("recon", "manifold", "ignore", "fro", "obj")])
        return U, V, np.array(parts)

    def restrict(self, V, cands):
        if self.mod is None:
            return self.O.restrict(V, self.tables, cands)
        return self.mod.restrict(V, self.Ls, cands, self.tables.supports)


def full_candidates(k, P):
    return {kk: [(p, 1) for p in range(P)] for kk in range(k)}


def cpu_sample(cpu, X, U0, V0, active, n_inner, gamma, delta, norm_X):
    """One bounded sample of an outer iteration on the CPU: `n_inner` inner steps + one `restrict` over all candidates.
    Returns the results (the parity check uses them) and the timings."""
    t0 = time.perf_counter()
    U, V, parts = cpu.inner_steps(X, U0.copy(), V0.copy(), active, n_inner, gamma, delta, norm_X)
    t_inner = (time.perf_counter() - t0) / n_inner
    t0 = time.perf_counter()
    surv = cpu.restrict(V, full_candidates(V.shape[1], len(cpu.tables)))
    t_restrict = time.perf_counter() - t0
    return {"U": U, "V": V, "parts": parts, "survivors": {kk: [int(p) for p, _ in v] for kk, v in surv.items()},
            "scores": {kk: [float(s) for _, s in v] for kk, v in surv.items()},
            "s_per_inner_step": t_inner, "s_restrict": t_restrict}


def run_reference_arm(a):
    """`--impl reference`: the reference's CPU implementation of the path on all host cores of the box.  A step is a
    bounded sample of one outer iteration at the FULL shape: `n_inner` of its 10 inner steps (update + objective)
    plus its one `restrict` over all candidates, n_inner sized from the first warm-up step so that the whole run fits
    `--ref-budget-s`; `value` scales the measured inner-step time to 10 steps (the 10 are identical work), while
    `ms_per_step` is the wall time actually spent per sample."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    use_all_cores()
    X = host_rows(0, a.m, a.n)
    Gs, nodelist, _ = make_pathways(a)
    cpu = CpuReference(Gs, nodelist, a.k)
    U0, V0 = initial_UV(a)
    norm_X = float(np.linalg.norm(X))
    gamma, delta = norm_X / a.k, 10 / norm_X
    active = [kk % a.pathways for kk in range(a.k)]
    total = a.warmup + a.steps
    n_inner = 1
    t_in, t_re, wall = [], [], []
    for s in range(total):
        t0 = time.perf_counter()
        r = cpu_sample(cpu, X, U0, V0, active, n_inner, gamma, delta, norm_X)
        dt = time.perf_counter() - t0
        if s == 0:      # size the sample: the remaining steps share what is left of the budget
            left = max(1.0, a.ref_budget_s - (time.perf_counter() - T_START))
            per_step = left / max(1, total - 1)
            n_inner = int(max(1, min(MODULUS, (per_step - r["s_restrict"]) // max(1e-9, r["s_per_inner_step"]))))
        if s >= a.warmup:
            t_in.append(r["s_per_inner_step"]); t_re.append(r["s_restrict"]); wall.append(dt)
    t_outer = MODULUS * float(np.mean(t_in)) + float(np.mean(t_re))
    value = 1.0 / t_outer
    cores = host_threads()
    sample = ("%d of the 10 inner steps + the restrict of one outer iteration per step, at the full shape, by %s; "
              "value = 1 / (10 x mean inner-step time + mean restrict time); ms_per_step is the wall time of a sample"
              % (n_inner, "the unmodified reference functions (baseline/_ref)" if cpu.kind == "reference" else "the oracle port"))
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": a.gpus,
        "steps": len(wall), "warmup": a.warmup, "ms_per_step": 1000.0 * float(np.mean(wall)), "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": config_dict(a),
        "ms_per_outer_iteration": 1000.0 * t_outer,
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": cpu.kind, "sample": sample,
                         "inner_steps_per_sample": n_inner, "s_per_inner_step": float(np.mean(t_in)),
                         "s_restrict": float(np.mean(t_re)), "s_tables": cpu.t_tables},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
def rel_err(got, want):
    got, want = np.asarray(got, dtype=np.float64), np.asarray(want, dtype=np.float64)
    denom = np.maximum(np.abs(want), 1e-300)
    return float(np.max(np.abs(got - want) / denom)) if got.size else 0.0


def run_ours(a):
    import torch
    from prmf_b200 import CudaEngine
    from prmf_b200.dist import DistContext, row_block
    from prmf_b200.engine import attach_collectives
    from prmf_b200.solver import init_latent_to_pathway_data, restrict_from_tables, sample_active

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback")
    ctx = DistContext.from_env()
    if ctx.world != a.gpus:
        raise SystemExit("bench.py: --gpus %d but WORLD_SIZE=%d (launch with torch.distributed.run)" % (a.gpus, ctx.world))
    dev = ctx.local_rank if ctx.world > 1 else 0
    torch.cuda.set_device(dev)
    sampler = ClockSampler(dev)
    sampler.start()                      # nvidia-smi needs ~1 s to come up: start it before the data setup
    stream = torch.cuda.Stream(device=dev)
    lo, hi = row_block(a.m, ctx.world, ctx.rank)
    m_local = hi - lo
    Gs, nodelist, packed = make_pathways(a)

    tf32 = a.x_dtype == "tf32"
    xdt = torch.float32 if tf32 else torch.float64
    xnp = np.float32 if tf32 else np.float64
    xsz = 4 if tf32 else 8
    Xh = None
    if a.x_gen == "host":
        Xh = torch.empty((m_local, a.n), dtype=xdt, pin_memory=True)
        host_rows(lo, hi, a.n, xnp, out=Xh.numpy())
        Xsrc = Xh.numpy()
    else:
        Xsrc = device_rows(lo, hi, a.n, xdt)
    eng = CudaEngine(m_local, a.m, a.n, a.k, device=dev, stream=stream.cuda_stream, x_dtype=a.x_dtype)
    attach_collectives(eng, ctx)
    eng.set_X(Xsrc)
    if a.x_gen == "device":
        del Xsrc
        torch.cuda.empty_cache()
    eng.set_pathways(packed)
    normX = float(np.sqrt(eng.normX_sq))
    gamma, delta = normX / a.k, 10 / normX

    U0, V0 = initial_UV(a)
    eng.set_UV(U0[lo:hi], V0)
    full_cands = init_latent_to_pathway_data(a.k, packed.P)

    host_t = [0.0]

    def outer_iteration():
        t0 = time.perf_counter()
        active = sample_active(full_cands, a.k)
        eng.set_active(active)
        t1 = time.perf_counter()
        eng.step_async(MODULUS, gamma, delta)
        # score tables enqueued behind the 10 steps, one host wait; the next block's X.V pass is already
        # streaming while the host runs restrict and the multinomial draws (as prmf_b200.nmf_pathway does)
        parts, _, _, (mass, qn, _) = eng.block_end(MODULUS, want_scores=True, prefetch=True)
        t2 = time.perf_counter()
        surv = restrict_from_tables(mass, qn, full_cands)
        host_t[0] += (t1 - t0) + (time.perf_counter() - t2)
        return parts, mass, qn, surv

    def sync_all():
        if ctx.world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if ctx.world == 1:
            return x
        import torch.distributed as dist
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    np.random.seed(1)                    # the multinomial draws of the timed loop: the same stream on every rank
    for _ in range(a.warmup):            # NOTE: the same number of steps on every rank (each holds collectives)
        outer_iteration()
    launches0 = eng.launch_count
    sync_all()
    sampler.mark_begin()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    # ---- timed region: exactly K steps, device events on the launching stream, max over ranks ----
    host_t[0] = 0.0
    e0.record(stream)
    for _ in range(a.steps):
        last = outer_iteration()
    e1.record(stream)
    sync_all()
    host_ms = host_t[0] * 1e3 / a.steps      # sampling + set_active + scores + restrict per outer iteration
    ms = e0.elapsed_time(e1)
    launches = eng.launch_count - launches0
    final_obj = float(last[0][-1, 4])
    if a.dump_outputs:
        dump_outputs(a, ctx, eng, lo, hi, last, packed.P)
    # ---- the same K steps again with an event pair around every phase of every inner step (the per-kernel
    #      durations of the roofline; the event records cost a few %, so they are kept out of `value`) ----
    eng.kernel_times(reset=True)
    eng.set_profiling(True)
    p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    p0.record(stream)
    for _ in range(a.steps):
        outer_iteration()
    p1.record(stream)
    sync_all()
    eng.set_profiling(False)
    clocks = sampler.stop()
    ms_profiled = p0.elapsed_time(p1) / a.steps
    kt = eng.kernel_times(reset=True)
    ms = max_over_ranks(ms)
    ms_per_step = ms / a.steps
    value = 1000.0 / ms_per_step

    # ---- roofline of the X-stream kernels (algorithmic bytes per launch / mean launch duration) ----
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s"
    wsz = 4 if tf32 else 8                      # bytes per element of the W operand (fp32 transposed copy in tf32 mode)
    bytes_xv = m_local * a.n * xsz + a.n * a.k * wsz + m_local * a.k * 8
    bytes_xtu = m_local * a.n * xsz + m_local * a.k * wsz + a.n * a.k * 8
    phase_ms = {name: (tot / max(1, cnt)) for name, (tot, cnt) in kt.items()}
    xv_ms, xtu_ms = phase_ms["xv"], phase_ms["xtu"]
    ach_xv = bytes_xv / (xv_ms * 1e-3) / 1e9 if xv_ms > 0 else 0.0
    ach_xtu = bytes_xtu / (xtu_ms * 1e-3) / 1e9 if xtu_ms > 0 else 0.0
    step_bytes = bytes_xv + bytes_xtu
    inner_ms = ms_per_step / MODULUS
    kname = "tc_rowdot_kernel" if tf32 else "skinny_tma_kernel" if a.k <= 10 else "skinny_tma_gen_kernel"
    dominant = kname + (" pass 2 (X^T.U)" if xtu_ms >= xv_ms else " pass 1 (X.V)")
    ach = ach_xtu if xtu_ms >= xv_ms else ach_xv
    traffic, traffic_src = ncu_traffic(kname, a, ctx.world)
    flops_pass = 2.0 * m_local * a.n * a.k
    roofline = {
        "bound": "hbm", "kernel": dominant, "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
        "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
        "note": ("launch durations come from a second, event-instrumented pass (an event pair around every launch makes "
                 "the step a few % slower than the timed pass); at k <= 10 the X-stream launches also contain the fused "
                 "U / V-update tails, so `frac` is a lower bound for the stream itself; inner_step.frac is the whole "
                 "timed step against the two-stream roofline"),
        "xv": {"ms": xv_ms, "GBps": ach_xv, "frac": ach_xv / peak, "bytes": bytes_xv},
        "xtu": {"ms": xtu_ms, "GBps": ach_xtu, "frac": ach_xtu / peak, "bytes": bytes_xtu},
        "inner_step": {"ms": inner_ms, "bytes": step_bytes, "GBps": step_bytes / (inner_ms * 1e-3) / 1e9,
                       "frac": step_bytes / (inner_ms * 1e-3) / 1e9 / peak,
                       "x_stream_share_of_step": (xv_ms + xtu_ms) / inner_ms if inner_ms > 0 else None,
                       "phase_ms": phase_ms, "host_ms_per_outer": host_ms,
                       "ms_per_outer_with_phase_events": ms_profiled},
    }
    if not tf32 and a.k > 10:
        # 2k flop per 8-byte element of X: above the fp64 ridge (~5 flop/B) the stream is DFMA-issue bound, not HBM bound
        tf = max(xv_ms, xtu_ms)
        roofline["fp64"] = {"flop_per_pass": flops_pass, "achieved_tflops": flops_pass / (tf * 1e-3) / 1e12 if tf > 0 else 0.0,
                            "peak_tflops": FP64_DFMA_PEAK_TFLOPS, "peak_source": "tools/fp64_microbench.cu (DFMA, measured)",
                            "frac": flops_pass / (tf * 1e-3) / 1e12 / FP64_DFMA_PEAK_TFLOPS if tf > 0 else 0.0,
                            "note": "arithmetic intensity %.1f flop/B: the binding limit at this k is the FP64 pipe" % (2.0 * a.k / 8)}

    # ---- parity: two inner steps + restrict from fixed U0 / V0, GPU (this run) vs the CPU reference on rank 0 ----
    parity, cpu = None, None
    if not a.no_parity:
        parity, cpu = parity_block(a, ctx, eng, Xh, lo, hi, Gs, nodelist, packed, U0, V0, gamma, delta, normX)

    # ---- e2e: the same outer iteration with HOST buffers (pinned X, U, V in; U, V, objective out) ----
    e2e = None
    if not a.no_e2e and Xh is not None:
        Uh = torch.empty((m_local, a.k), dtype=torch.float64, pin_memory=True)
        Vh = torch.empty((a.n, a.k), dtype=torch.float64, pin_memory=True)
        Uh.copy_(torch.from_numpy(np.ascontiguousarray(U0[lo:hi]))); Vh.copy_(torch.from_numpy(V0))
        Xn, Un, Vn = Xh.numpy(), Uh.numpy(), Vh.numpy()

        # Every step uploads its X from pinned host memory (H2D inside the timed region) -- into one of two device staging
        # buffers on a copy stream, so that the upload of step i+1 overlaps the compute of step i (the first upload is
        # exposed and counted); the engine then takes the staged block (device-to-device + transposed copy), runs the
        # step and the result is read back.
        copy_stream = torch.cuda.Stream(device=dev)
        stage = [torch.empty((m_local, a.n), dtype=xdt, device="cuda") for _ in range(2)]
        staged = [torch.cuda.Event(), torch.cuda.Event()]

        def start_upload(i):
            with torch.cuda.stream(copy_stream):
                stage[i % 2].copy_(Xh, non_blocking=True)
                staged[i % 2].record(copy_stream)

        def e2e_iteration(i, last):
            staged[i % 2].synchronize()         # this step's X has arrived
            if not last:
                start_upload(i + 1)             # the next step's upload runs under this step's compute
            eng.set_X(stage[i % 2])
            eng.set_UV(Un, Vn)
            active = sample_active(full_cands, a.k)
            eng.set_active(active)
            eng.step_async(MODULUS, gamma, delta)
            p, _, _, (mass, qn, _) = eng.block_end(MODULUS, want_scores=True, prefetch=False)
            restrict_from_tables(mass, qn, full_cands)
            Uo, Vo = eng.get_UV()               # D2H of the result
            return float(p[-1, 4]), Uo, Vo

        n_e2e = max(2, a.steps)
        start_upload(0); e2e_iteration(0, True)                      # warm-up
        sync_all()
        t0 = time.perf_counter()
        e0.record(stream)
        start_upload(0)
        for i in range(n_e2e):
            e2e_iteration(i, i == n_e2e - 1)
        e1.record(stream)
        sync_all()
        wall_ms = (time.perf_counter() - t0) * 1e3 / n_e2e
        ems = max_over_ranks(wall_ms)           # wall clock: the copy stream's work is part of the step
        del stage
        e2e = {"value": 1000.0 / ems, "unit": UNIT, "ms_per_step": ems,
               "h2d_bytes_per_step": int(m_local * a.n * xsz + (m_local + a.n) * a.k * 8),
               "d2h_bytes_per_step": int((m_local + a.n) * a.k * 8 + MODULUS * 64 + 2 * a.k * packed.P * 8),
               "steps": n_e2e,
               "note": "X of every step uploaded from pinned host memory (double-buffered: the upload of step i+1 overlaps "
                       "the compute of step i, the first one is exposed), U / V in and out, objective out; PCIe-bound"}

    # ---- time to converge: the public entry point on the planted instance, host arrays in and out ----
    ttc = None
    if not a.no_converge and Xh is not None:
        ttc = time_to_converge(a, ctx, Xh.numpy(), lo, Gs, nodelist, packed, value, eng if ctx.world > 1 else None)

    exch_mode = eng.exchange_mode
    ctx.barrier()
    eng.close()
    if ctx.rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps,
            "warmup": a.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f64" if not tf32 else "tf32 X products (fp32 accumulate), f64 updates",
            "data": "synthetic", "config": config_dict(a),
            "parallelism": "rows of X,U sharded over %d GPU(s)" % a.gpus + (
                "" if a.gpus == 1 else (", per-step sum over ranks of [X^T U | U^T U]: " + {
                    "nccl": "ncclAllReduce", "p2p-v-update": "NVLink peer loads fused into the V-update kernel",
                    "p2p-pass2": "NVLink peer exchange fused into the pass-2 X-stream kernel (exchange + V update)",
                    "p2p-push-block": "NVLink peer stores (push) inside the persistent step kernel, summed in rank order from local memory",
                    "none": "none"}.get(exch_mode, exch_mode))),
            "inner_steps_per_s": 1000.0 / inner_ms,
            "roofline": roofline, "cpu_baseline": cpu, "parity": parity, "e2e": e2e, "time_to_converge": ttc,
            "gpu_launches": int(launches), "clocks": clocks, "final_obj": final_obj,
        }
        print(json.dumps(line))
    if ctx.world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()


def ncu_traffic(kname, a, world):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, from the committed ncu summary
    (profiles/ncu_traffic.json, written by tools/ncu_summary.py from a `ncu --set full` capture of this command)."""
    try:
        table = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
    except Exception:
        return None, "profiles/ncu_traffic.json not found"
    key = "%s|m=%d|n=%d|k=%d|gpus=%d" % (kname, a.m, a.n, a.k, world)
    ent = table.get(key)
    if not ent:
        return None, "no ncu capture for %s in profiles/ncu_traffic.json" % key
    return float(ent["dram_bytes_per_launch"]), ent.get("source", "profiles/ncu_traffic.json")


def parity_block(a, ctx, eng, Xh, lo, hi, Gs, nodelist, packed, U0, V0, gamma, delta, normX):
    """Two inner steps + scores/restrict from fixed inputs on the GPU path; rank 0 repeats them with the CPU reference
    on the full-shape arrays (all host cores) and reports max relative errors.  The same CPU computation is the
    `cpu_baseline` timing at N = 1.  Digests of V must agree on all ranks (bitwise) and, like the printed objective
    parts, across N."""
    from prmf_b200.solver import init_latent_to_pathway_data, restrict_from_tables
    n_inner = a.cpu_inner_steps
    active = [kk % a.pathways for kk in range(a.k)]
    eng.set_UV(U0[lo:hi], V0)
    eng.set_active(active)
    parts, _, _ = eng.step(n_inner, gamma, delta)
    Ug, Vg = eng.get_UV()
    mass, qn, _ = eng.scores()
    surv = restrict_from_tables(mass, qn, init_latent_to_pathway_data(a.k, packed.P))
    surv_ids = {kk: [int(p) for p, _ in v] for kk, v in surv.items()}
    surv_scores = {kk: [float(s) for _, s in v] for kk, v in surv.items()}
    v_digests = ctx.all_gather_bytes(digest(Vg).encode())
    U_full = ctx.all_gather_rows(Ug, a.m)
    out = {"inner_steps": n_inner, "active": "factor f -> pathway f",
           "gpu_obj_parts": parts[:, :5].tolist(), "gpu_V_sha256_16": v_digests[0].decode(),
           "gpu_U_sha256_16": digest(U_full), "ranks_bitwise_equal_V": len(set(v_digests)) == 1,
           "gpu_survivors_sha256_16": hashlib.sha256(json.dumps(surv_ids, sort_keys=True).encode()).hexdigest()[:16],
           "gpu_survivors_per_factor": [len(surv_ids[kk]) for kk in sorted(surv_ids)]}
    cpu = None
    if ctx.rank == 0 and not a.no_cpu_baseline and a.m * a.n > (1 << 29):
        out["subsample"] = parity_subsample(a, eng, Gs, nodelist, packed, U0, V0)
    if ctx.rank == 0 and not a.no_cpu_baseline and a.m * a.n <= (1 << 29):
        use_all_cores()
        X = Xh.numpy() if (ctx.world == 1 and Xh is not None and Xh.dtype.is_floating_point and Xh.element_size() == 8) \
            else host_rows(0, a.m, a.n)
        if a.x_dtype == "tf32":            # the CPU side sees the X the device holds (rounded to tf32 at store time)
            sys.path.insert(0, os.path.join(ROOT, "tests"))
            from helpers import tf32_round
            X = tf32_round(X.astype(np.float32))
        ref = CpuReference(Gs, nodelist, a.k)
        r = cpu_sample(ref, np.asarray(X, dtype=np.float64), U0, V0, active, n_inner, gamma, delta, normX)
        same = all(surv_ids[kk] == r["survivors"][kk] for kk in surv_ids)
        out.update({
            "vs": "unmodified reference functions (baseline/_ref: nmf_manifold_vec_update, restrict)" if ref.kind == "reference"
                  else "oracle port (oracle/prmf_oracle.py)",
            "U_max_rel_err": rel_err(U_full, r["U"]), "V_max_rel_err": rel_err(Vg, r["V"]),
            "obj_parts_max_rel_err": rel_err(parts[:, :5], r["parts"]),
            "restrict_survivors_identical": bool(same),
            "restrict_scores_max_rel_err": max(rel_err(surv_scores[kk], r["scores"][kk]) for kk in surv_ids) if same else None,
            "tolerance": "fp64 mode: obj parts 1e-9, U/V 1e-8 over the two steps (SURVEY 8c)" if a.x_dtype == "f64"
                         else "tf32 mode: objective parts and U/V 1e-3 (tests/test_tf32.py; not the parity mode)"})
        t_outer = MODULUS * r["s_per_inner_step"] + r["s_restrict"]
        if ctx.world == 1:
            cpu = {"value": 1.0 / t_outer, "unit": UNIT, "cores": host_threads(), "kind": ref.kind,
                   "sample": "%d inner steps + 1 restrict at the full shape by %s, inner-step time scaled to 10" % (
                       n_inner, "the unmodified reference functions (baseline/_ref)" if ref.kind == "reference" else "the oracle port"),
                   "s_per_inner_step": r["s_per_inner_step"], "s_restrict": r["s_restrict"], "s_tables": ref.t_tables}
    ctx.barrier()
    return out, cpu


def parity_subsample(a, eng_big, Gs, nodelist, packed, U0, V0, rows=2048):
    """Instances too large for a CPU run at full shape (config 5): the first `rows` samples of the same matrix on a second,
    single-GPU engine of the same mode against the CPU reference on those rows (SURVEY 8d: a row subsample)."""
    import torch
    from prmf_b200 import CudaEngine
    from prmf_b200.solver import init_latent_to_pathway_data, restrict_from_tables
    rows = min(rows, a.m)
    tf32 = a.x_dtype == "tf32"
    Xs = (device_rows(0, rows, a.n, torch.float32 if tf32 else torch.float64) if a.x_gen == "device"
          else torch.from_numpy(host_rows(0, rows, a.n, np.float32 if tf32 else np.float64)).cuda())
    active = [kk % a.pathways for kk in range(a.k)]
    with CudaEngine(rows, rows, a.n, a.k, device=torch.cuda.current_device(), x_dtype=a.x_dtype) as eng:
        eng.set_X(Xs)
        eng.set_pathways(packed)
        normX = float(np.sqrt(eng.normX_sq))
        gamma, delta = normX / a.k, 10 / normX
        eng.set_UV(U0[:rows], V0)
        eng.set_active(active)
        parts, _, _ = eng.step(a.cpu_inner_steps, gamma, delta)
        Ug, Vg = eng.get_UV()
        mass, qn, _ = eng.scores()
    surv = restrict_from_tables(mass, qn, init_latent_to_pathway_data(a.k, packed.P))
    surv_ids = {kk: [int(p) for p, _ in v] for kk, v in surv.items()}
    X = Xs.cpu().numpy().astype(np.float64)
    if tf32:
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        from helpers import tf32_round
        X = tf32_round(X.astype(np.float32))
    use_all_cores()
    ref = CpuReference(Gs, nodelist, a.k, force_port=True)       # the port: 2 000 n x n DOK matrices take minutes to build
    r = cpu_sample(ref, X, U0[:rows], V0, active, a.cpu_inner_steps, gamma, delta, normX)
    same = all(surv_ids[kk] == r["survivors"][kk] for kk in surv_ids)
    return {"rows": rows, "vs": "oracle port (oracle/prmf_oracle.py) on the first %d samples" % rows,
            "U_max_rel_err": rel_err(Ug, r["U"]), "V_max_rel_err": rel_err(Vg, r["V"]),
            "obj_parts_max_rel_err": rel_err(parts[:, :5], r["parts"]), "restrict_survivors_identical": bool(same),
            "tolerance": "tf32 mode: objective parts and U/V 1e-3 (tests/test_tf32.py; not the parity mode)" if tf32 else "fp64: 1e-9 / 1e-8"}


def time_to_converge(a, ctx, X_local, lo, Gs, nodelist, packed, steady_value, shared_engine=None):
    """BASELINE.json's second metric: `nmf_pathway` (host arrays in, host arrays out) on the planted instance until the
    loop guard exits (tol 1e-3, :715,:772-774).  The X block is modified in place (planted bumps).  On several GPUs
    the solves run on the bench's own engine (`engine_factory`), as a caller that solves more than once would: creating
    the NCCL communicator and mapping the peer buffers costs seconds and is not part of the path."""
    from prmf_b200 import nmf_pathway
    plant_signal(X_local, Gs, lo, a.m)
    times, info = [], None
    kw = {}
    if shared_engine is not None:
        class _Keep:                              # nmf_pathway closes the engine it was given; keep ours for the second solve
            def __init__(self, eng): self._e = eng
            def __getattr__(self, name): return getattr(self._e, name)
            def close(self): pass
        kw["engine_factory"] = lambda *args, **kwargs: _Keep(shared_engine)
    for rep in range(2):                        # the first call also pays one-off costs (lazy kernel loading)
        np.random.seed(1)
        trace = {"keep_blocks": 0}
        with contextlib.redirect_stderr(io.StringIO()):
            ctx.barrier()
            t0 = time.perf_counter()
            U, V, od = nmf_pathway(X_local, packed, k_latent=a.k, nodelist=nodelist, quiet=True, x_dtype=a.x_dtype,
                                   ctx=ctx, X_is_local=True, m_global=a.m, trace=trace, **kw)
            times.append(time.perf_counter() - t0)
        n_inner = len(trace["obj_parts"])
        fmap = {int(kk): [int(p) for p, _ in v] for kk, v in od["latent_to_pathway_data"].items()}
        info = {"inner_steps": n_inner, "outer_iterations": n_inner // MODULUS, "final_obj": float(od["obj"]),
                "assignment": [fmap[kk][0] if len(fmap[kk]) == 1 else fmap[kk] for kk in sorted(fmap)],
                "V_sha256_16": digest(V)}
    steady = info["outer_iterations"] / steady_value
    info.update({"seconds": times[1], "seconds_first_call": times[0], "tol": 1e-3,
                 "instance": "the bench instance with a rank-1 bump planted on the genes of 10 pathways (SURVEY 8d)",
                 "includes": ("engine creation, " if shared_engine is None else "(engine and communicators reused) ") +
                             "X upload + transposed copy, the whole loop, download of U and V "
                             "(pathways pre-packed; no file I/O, no quantile_transform)",
                 "steady_state_seconds": steady, "ratio_to_steady_state": times[1] / steady if steady > 0 else None})
    return info


T_START = time.perf_counter()

if __name__ == "__main__":
    import faulthandler
    args = parse_args()
    # never hang a GPU box: die loudly instead (the CPU reference arm legitimately runs for minutes)
    faulthandler.dump_traceback_later(900 if args.impl == "reference" else 600, exit=True)
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_ours(args)
