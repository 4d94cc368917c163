"""Bit-exact tests of the X-stream products X.V (pass 1, `prmf_project`) and X^T.U (pass 2, `prmf_project_t`).

X, U and V hold small nonzero integers (uniform on 1..7).  Every product and partial sum is then an integer far below
2^53, so the fp64 kernels must return exactly the int64 product whatever their summation order, chunking or tiling;
one dropped or repeated term moves an entry by at least 1.  The same holds in tf32 mode: integers below 2^11 are exact
in tf32, and the fp32 accumulation of a chunk stays exact while its partial sums stay below 2^24.

The first half asks the library's launch planner (`prmf_plan_xstream`, the one `prmf_create_ex` runs) for the plan of
every handle in the shape table below and checks, without a GPU, that the table reaches the edges where a stream kernel
can go wrong (empty chunks, ragged stages, narrow last panels, idle factor groups) and that no kernel reads W outside its
shared-memory slot.  The GPU tests then run every kernel instantiation over that table and compare bitwise.
"""
import numpy as np
import pytest

from helpers import xstream_plan

B200_SMS = 148          # the table proves its regimes for this SM count only
RS = 8                  # stage height (rows) of the TMA kernels, kTmaRS in kernels.cuh
RING_LIMIT = 220 * 1024  # a PRMF_TMA_STAGES ring above this size gives way to the default stage count

# (m, n) shapes: pass 1 streams Xt (rows = n, cols = m), pass 2 streams X (rows = m, cols = n)
SHAPES = [(1, 1), (5, 33), (37, 131), (1000, 6750), (1025, 1000), (2049, 33), (3, 4100), (300, 257), (993, 520),
          (4500, 1031)]
K_SKINNY = list(range(1, 11))                                     # skinny_tma_kernel<K, 8, 0>
K_GEN = [11, 13, 17, 25, 33, 49, 65, 66, 97, 98, 128]              # skinny_tma_gen_kernel<KT, FG>
K_TF32 = [1, 10, 16, 17, 64, 100, 128]
TF32_SHAPES = [(1, 1), (5, 33), (37, 131), (300, 257), (2049, 33), (1000, 6750), (4500, 1031)]
# launch switches (read when a handle is created) and the k they run with
SWITCH_CASES = [
    ({"PRMF_TMA_STAGES": "2"}, K_SKINNY + K_GEN),
    ({"PRMF_TMA_STAGES": "12"}, [97]),
    ({"PRMF_TMA_STAGES": "12"}, [10]),       # the 12-stage ring fits narrow panels only: the other handles keep 3 stages
    ({"PRMF_TMA_STAGES": "12"}, [25]),       # the same for the general-k kernel (FG = 2: 4 stages by default)
]
SWITCH_IDS = ["stages2", "stages12", "stages12_fallback_skinny", "stages12_fallback_gen"]


# ---- the plan, and what the general-k kernel reads ---------------------------------------------------------------
def fg_kt(k):
    """(FG, KT) of the general-k kernel a handle with k > 10 factors runs."""
    plan = xstream_plan(1, 1, k)
    return plan.fg, plan.kt


def w_slot_bytes(k, kt):
    """Bytes the general-k kernel reserves for one stage's W rows, kernels.cuh `w_slot`."""
    return ((RS * k + kt) * 8 + 127) & ~127


def kernel_of(k):
    """Name of the X-stream kernel an fp64 handle with k factors runs."""
    if k > 10:
        return "skinny_tma_gen_kernel<%d,%d>" % fg_kt(k)[::-1]
    return "skinny_tma_kernel<%d,%d,0>" % (k, RS)


def pass_regimes(cols, rows, p, fg):
    """The edges one pass meets: the row chunks and column panels of its launch, as the kernels see them."""
    out = set()
    out.add("one panel" if p.panels == 1 else "several panels")
    if cols - (p.panels - 1) * p.panel_w < p.panel_w:             # the rest of its width is zero pad columns
        out.add("narrow last panel")
    if cols % 4:
        out.add("cols % 4 != 0")
    if cols == 1:
        out.add("cols == 1")
    if rows == 1:
        out.add("rows == 1")
    if rows < RS:
        out.add("rows < RS")
    if p.chunks == 1:
        out.add("one chunk")
    for c in range(p.chunks):
        beg, end = c * p.rows_per_chunk, min(rows, (c + 1) * p.rows_per_chunk)
        if end <= beg:
            out.add("empty chunk")
        elif (end - beg) % RS:
            out.add("ragged last stage")
    if p.panels > 1:
        out.add("several panels at FG %d" % fg)
    return out


def regimes(m, n, k):
    """{"pass 1": set, "pass 2": set} for an fp64 TMA handle."""
    plan = xstream_plan(m, n, k)
    return {"pass 1": pass_regimes(m, n, plan.pass1, plan.fg), "pass 2": pass_regimes(n, m, plan.pass2, plan.fg)}


def max_w_index(k, fg, kt, clamped=True):
    """Largest W index (in doubles from the start of a stage's W slot) that skinny_tma_gen_kernel reads: factor group g
    reads sw[f + r*k + c] for r < RS, c < KT, where f = g*KT, or 0 for a group whose factors all lie at or beyond k
    (kernels.cuh, `fr`).  `clamped=False` models a loop in which every group reads its own columns."""
    first = [g * kt if (g * kt < k or not clamped) else 0 for g in range(fg)]
    return max(first) + (RS - 1) * k + kt - 1


# ---- CPU checks of the table ----------------------------------------------------------------------------------
REQUIRED = ["one panel", "several panels", "narrow last panel", "cols % 4 != 0", "cols == 1", "rows == 1",
            "rows < RS", "one chunk", "ragged last stage", "empty chunk"]


def test_shape_table_covers_the_launch_plan_edges():
    for pas in ("pass 1", "pass 2"):
        seen = set()
        for m, n in SHAPES:
            for k in K_SKINNY + K_GEN:
                seen |= regimes(m, n, k)[pas]
        missing = [r for r in REQUIRED + ["several panels at FG %d" % fg for fg in (1, 2, 4, 8)] if r not in seen]
        assert not missing, "%s never meets %s" % (pas, missing)


def test_every_instantiation_meets_an_empty_chunk_a_ragged_stage_and_a_narrow_panel():
    by_kernel = {}
    for m, n in SHAPES:
        for k in K_SKINNY + K_GEN:
            r = regimes(m, n, k)
            d = by_kernel.setdefault(kernel_of(k), {"pass 1": set(), "pass 2": set()})
            for pas in d:
                d[pas] |= r[pas]
    want = {"skinny_tma_kernel<%d,8,0>" % k for k in K_SKINNY} | \
           {"skinny_tma_gen_kernel<%d,%d>" % (kt, fg) for fg, kt in {fg_kt(k) for k in range(11, 129)}}
    assert set(by_kernel) == want
    for name, d in sorted(by_kernel.items()):
        for pas, seen in d.items():
            for r in ("empty chunk", "ragged last stage", "narrow last panel"):
                assert r in seen, "%s never meets %r in %s" % (name, r, pas)


def test_general_k_choices_reach_idle_and_ragged_factor_groups():
    """K_GEN holds a ragged last group (k = 25: 16 + 9), wholly idle groups (k = 66, 98: the worst W over-reads
    of the unclamped loop) and the FG = 4 idle group (k = 33)."""
    assert fg_kt(25) == (2, 16) and 25 % 16
    assert fg_kt(33) == (4, 12) and 3 * 12 >= 33
    assert fg_kt(66) == (8, 12) and sum(g * 12 >= 66 for g in range(8)) == 2
    assert fg_kt(98) == (8, 16) and 7 * 16 >= 98
    # every (FG, KT) that k = 11..128 can select: the library instantiates exactly these (tests/test_sass.py)
    assert {fg_kt(k) for k in range(11, 129)} == {(1, 12), (1, 16), (2, 12), (2, 16), (4, 12), (4, 16), (8, 12), (8, 16)}


@pytest.mark.parametrize("k", range(11, 129))
def test_general_k_kernel_reads_w_inside_its_slot(k):
    """The largest W index read lies inside the W slot, and the kernel's stage layout (x rows + w_slot, then 2
    mbarriers per stage) lies inside the ring the host sizes, for every PRMF_TMA_STAGES a handle can be given, at the
    narrowest panel (n = 1: 4 columns) and the widest (n = 1024: 1024 / FG columns)."""
    fg, kt = fg_kt(k)
    slot = w_slot_bytes(k, kt) // 8
    assert max_w_index(k, fg, kt) <= RS * k + kt - 2 < slot
    for stages in range(2, 13):
        for n in (1, 1024):
            plan = xstream_plan(1, n, k, stages=stages)
            p = plan.pass2
            kernel_end = plan.stages * (RS * p.panel_w * 8 + w_slot_bytes(k, kt)) + 2 * plan.stages * 8
            assert kernel_end <= p.ring_smem


def test_w_slot_check_flags_the_unclamped_loop():
    """If every group read its own columns, the last row of the last stage would read past the W slot at k = 66 and 98
    and, at the default 6 stages, 16 bytes past the end of the shared memory the host requests."""
    for k in (66, 98):
        fg, kt = fg_kt(k)
        plan = xstream_plan(1000, 6750, k)
        p = plan.pass2                                           # 6750 genes: panels of the widest width, 128 columns
        last = max_w_index(k, fg, kt, clamped=False)
        assert last >= w_slot_bytes(k, kt) // 8
        x_stage = RS * p.panel_w * 8
        end_of_read = (plan.stages - 1) * (x_stage + w_slot_bytes(k, kt)) + x_stage + (last + 1) * 8
        assert end_of_read - p.ring_smem == 16
    bad = [k for k in range(11, 129) if max_w_index(k, *fg_kt(k), clamped=False) >= w_slot_bytes(k, fg_kt(k)[1]) // 8]
    assert {66, 98} <= set(bad) <= set(range(65, 79)) | set(range(97, 111))


def test_default_ring_fits_at_the_widest_panel():
    """An oversized PRMF_TMA_STAGES gives way to the default stage count, so the default ring must fit at every k."""
    for k in range(1, 129):
        plan = xstream_plan(1024, 1024, k)                      # 1024 columns: panels of 1024 / FG columns
        assert max(plan.pass1.ring_smem, plan.pass2.ring_smem) <= RING_LIMIT, k


def test_switch_cases_reach_the_intended_kernels():
    for m, n in SHAPES:
        for k in K_SKINNY + K_GEN:
            assert xstream_plan(m, n, k, stages=2).stages == 2, (m, n, k)
        assert xstream_plan(m, n, 97, stages=12).stages == 12, (m, n)
    assert kernel_of(97) == "skinny_tma_gen_kernel<16,8>" and kernel_of(10) == "skinny_tma_kernel<10,8,0>"
    # at k = 10 and 25 a 12-stage ring fits narrow panels only: wider handles keep the default 3 / 4 stages
    for k, default in ((10, 3), (25, 4)):
        stages = {(m, n): xstream_plan(m, n, k, stages=12).stages for m, n in SHAPES}
        assert set(stages.values()) == {default, 12} and stages[(1000, 6750)] == default, k
    # PRMF_TMA_STAGES=2 wraps the mbarrier phase every two stages: some chunk of the table runs more than 2 stages
    plan = xstream_plan(1000, 6750, 66, stages=2)
    assert plan.stages == 2 and plan.pass2.rows_per_chunk > 4 * RS


def test_tf32_table_covers_the_tensor_core_edges():
    seen = set()
    for m, n in TF32_SHAPES:
        plan = xstream_plan(m, n, 16, x_dtype="tf32")
        for R, C, chunks in ((m, n, plan.tc_chunks1), (n, m, plan.tc_chunks2)):
            if R % 128:
                seen.add("rows % 128 != 0")
            if C % 32:
                seen.add("cols % 32 != 0")
            if C < 32:
                seen.add("cols < 32")
            if C >= 1024 and chunks > 1:
                seen.add("several column chunks")
    assert seen == {"rows % 128 != 0", "cols % 32 != 0", "cols < 32", "several column chunks"}
    kp = {-(-k // 16) * 16 for k in K_TF32}
    assert min(kp) == 16 and max(kp) == 128
    tcols = set()
    for k in kp:
        t = 32
        while t < k:
            t *= 2
        tcols.add(t)
    assert tcols == {32, 64, 128}


# ---- GPU: bitwise products --------------------------------------------------------------------------------------
def _ints(rng, *shape):
    return rng.integers(1, 8, size=shape).astype(np.float64)


def _operands(m, n, k, seed):
    rng = np.random.Generator(np.random.PCG64(seed))
    return _ints(rng, m, n), _ints(rng, m, k), _ints(rng, n, k)


def _exact(X, U, V):
    Xi, Ui, Vi = X.astype(np.int64), U.astype(np.int64), V.astype(np.int64)
    R = Xi - Ui @ Vi.T
    return Xi @ Vi, Xi.T @ Ui, int((Xi * Xi).sum()), int((R * R).sum())


@pytest.fixture(scope="module")
def b200():
    import torch
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    assert sms == B200_SMS, ("the shape table of this file proves its launch-plan edges for %d SMs; this device has %d"
                             % (B200_SMS, sms))
    return sms


def _check_products(eng, X, U, V, what, residual=True):
    A, B, nx2, r2 = _exact(X, U, V)
    np.testing.assert_array_equal(eng.project(), A, err_msg="X.V, " + what)
    np.testing.assert_array_equal(eng.project_t(), B, err_msg="X^T.U, " + what)
    assert eng.normX_sq == nx2, "||X||^2, " + what
    if residual:
        assert eng.residual_sq() == r2, "||X - U V^T||^2, " + what


def _run_products(m, n, ks, x_dtype="f64", residual=True, label=""):
    from prmf_b200 import CudaEngine
    for k in ks:
        X, U, V = _operands(m, n, k, seed=7 * m + 3 * n + k)
        with CudaEngine(m, m, n, k, x_dtype=x_dtype) as eng:
            eng.set_X(X)
            eng.set_UV(U, V)
            _check_products(eng, X, U, V, "%s m=%d n=%d k=%d %s" % (x_dtype, m, n, k, label), residual)


@pytest.mark.gpu
@pytest.mark.parametrize("m,n", SHAPES)
def test_products_bitwise_every_instantiation(b200, m, n):
    """Every skinny_tma_kernel<K,8,0> (k = 1..10) and every reachable skinny_tma_gen_kernel<KT,FG>, on every shape."""
    _run_products(m, n, K_SKINNY + K_GEN)


@pytest.mark.gpu
@pytest.mark.parametrize("env,ks", SWITCH_CASES, ids=SWITCH_IDS)
def test_products_bitwise_under_launch_switches(b200, monkeypatch, env, ks):
    """PRMF_TMA_STAGES=2: the ring wraps every two stages; PRMF_TMA_STAGES=12: skinny_tma_gen_kernel<16,8> with a
    12-stage ring at k = 97, and skinny_tma_kernel<10,8,0> / skinny_tma_gen_kernel<16,2> with 12 stages where that ring
    fits and the default stage count elsewhere.  test_switch_cases_reach_the_intended_kernels checks which stage count
    each handle runs."""
    for key, val in env.items():
        monkeypatch.setenv(key, val)
    for m, n in SHAPES:
        _run_products(m, n, ks, residual=False, label=str(env))


@pytest.mark.gpu
@pytest.mark.parametrize("m,n", TF32_SHAPES)
def test_tf32_products_bitwise(b200, m, n):
    """tcgen05 path: integer operands are exact in tf32 and their fp32 chunk sums stay below 2^24."""
    _run_products(m, n, K_TF32, x_dtype="tf32")


@pytest.mark.gpu
@pytest.mark.parametrize("x_dtype,k", [("f64", 6), ("f64", 25), ("tf32", 10), ("tf32", 17)])
def test_input_layouts_bitwise(b200, x_dtype, k):
    """Host column slices (ld > n), strided CUDA views, Fortran order and fp32 inputs store the same X."""
    import torch
    from prmf_b200 import CudaEngine
    m, n = 37, 131                                         # n not a multiple of 16
    X, U, V = _operands(m, n, k, seed=11 + k)
    wide = np.zeros((m, n + 21))
    wide[:, :n] = X
    wide[:, n:] = np.nan                                   # never read: the columns past n of each row
    flavours = {"host slice": wide[:, :n], "fortran": np.asfortranarray(X),
                "device slice": torch.from_numpy(wide).cuda()[:, :n], "device": torch.from_numpy(X).cuda()}
    if x_dtype == "tf32":
        w32 = wide.astype(np.float32)
        flavours.update({"f32 host": X.astype(np.float32), "f32 host slice": w32[:, :n],
                         "f32 device": torch.from_numpy(X.astype(np.float32)).cuda(),
                         "f32 device slice": torch.from_numpy(w32).cuda()[:, :n]})
    with CudaEngine(m, m, n, k, x_dtype=x_dtype) as eng:
        eng.set_UV(U, V)
        for name, Xf in flavours.items():
            eng.set_X(Xf)
            _check_products(eng, X, U, V, "%s %s k=%d" % (name, x_dtype, k))


@pytest.mark.gpu
@pytest.mark.parametrize("x_dtype,m,n,k", [("f64", 300, 257, 6), ("f64", 993, 520, 66), ("tf32", 300, 257, 17)])
def test_pooled_buffers_do_not_leak(b200, x_dtype, m, n, k):
    """A destroyed handle leaves X, its transposed copy and its arena (U, V, the chunk partials) to the next handle of
    the same shape.  Fill them with NaN first: none of it may reach the next handle's results."""
    from prmf_b200 import CudaEngine
    nan = np.full((m, n), np.nan)
    with CudaEngine(m, m, n, k, x_dtype=x_dtype) as eng:
        eng.set_X(nan)
        eng.set_UV(np.full((m, k), np.nan), np.full((n, k), np.nan))
        eng.project(); eng.project_t()
    X, U, V = _operands(m, n, k, seed=5)
    with CudaEngine(m, m, n, k, x_dtype=x_dtype) as eng:
        eng.set_X(X)
        eng.set_UV(U, V)
        _check_products(eng, X, U, V, "after a NaN handle, %s k=%d" % (x_dtype, k))


# ---- GPU: state interplay (fp64) --------------------------------------------------------------------------------
def _instance(m, n, k, P, seed):
    from prmf_b200 import pack_pathways, synth
    X, nodelist, Gs = synth.small_instance(m=m, n=n, k_true=min(3, P), n_pathways=P, pathway_size=12, seed=seed,
                                           weighted=True)
    rng = np.random.Generator(np.random.PCG64(seed + 100))
    U = 3 * (1 - rng.random((m, k)))
    V = 3 * (1 - rng.random((n, k)))
    active = [int(rng.integers(0, P)) for _ in range(k)]
    return X, pack_pathways(Gs, nodelist), U, V, active


def _close_products(eng, X):
    """project / project_t against numpy for the U, V the engine holds: |got - ref| <= 1e-13 (|X| |W|)."""
    U, V = eng.get_UV()
    A, B = eng.project(), eng.project_t()
    assert np.all(np.abs(A - X @ V) <= 1e-13 * (np.abs(X) @ np.abs(V)))
    assert np.all(np.abs(B - X.T @ U) <= 1e-13 * (np.abs(X).T @ np.abs(U)))


@pytest.mark.gpu
@pytest.mark.parametrize("k", [6, 12])
def test_projections_after_steps_and_speculative_pass(b200, k):
    from prmf_b200 import CudaEngine
    X, packed, U, V, active = _instance(300, 1200, k, 9, seed=40 + k)
    with CudaEngine(300, 300, 1200, k) as eng:
        eng.set_X(X); eng.set_pathways(packed); eng.set_UV(U, V); eng.set_active(active)
        eng.step(3, 2.0, 0.4)
        _close_products(eng, X)
        eng.step_async(2, 2.0, 0.4)
        eng.block_end(2, want_scores=True, prefetch=True)
        _close_products(eng, X)


@pytest.mark.gpu
@pytest.mark.parametrize("k", [6, 12])
def test_projections_between_blocks_are_bitwise_neutral(b200, k):
    """prmf_project uses the second U buffer and prmf_project_t the second V buffer as scratch: calling them between
    blocks (after a speculative pass, too) must not change any later step."""
    from prmf_b200 import CudaEngine
    X, packed, U, V, active = _instance(300, 1200, k, 9, seed=21)
    results = []
    for probe in (False, True):
        with CudaEngine(300, 300, 1200, k) as eng:
            eng.set_X(X); eng.set_pathways(packed); eng.set_UV(U, V)
            log = []
            for block in range(3):
                eng.set_active([(a + block) % 9 for a in active])
                eng.step_async(4, 2.0, 0.4)
                parts, _, _, tables = eng.block_end(4, want_scores=True, prefetch=block != 1)
                if probe:
                    eng.project(); eng.project_t()
                log.append((parts.copy(), tables[0].copy()) + eng.get_UV())
            parts, _, _ = eng.step(2, 2.0, 0.4)
            log.append((parts,) + eng.get_UV())
            results.append(log)
    for a, b in zip(*results):
        for x, y in zip(a, b):
            assert np.array_equal(x, y)


@pytest.mark.gpu
@pytest.mark.parametrize("k", [6, 12])
def test_set_X_after_speculative_pass(b200, k):
    """block_end(prefetch=True) then set_X(X2): the speculative pass over the old X is discarded.  The steps that follow
    are bitwise those of the same handle without the speculative pass, and match a fresh handle on X2 to rounding (a
    fresh handle recomputes V^T V from V in another summation order than the V update leaves it)."""
    from prmf_b200 import CudaEngine
    X, packed, U, V, active = _instance(300, 1200, k, 9, seed=61)
    X2 = np.random.Generator(np.random.PCG64(62)).random((300, 1200)) * 3
    runs = []
    for prefetch in (True, False):
        with CudaEngine(300, 300, 1200, k) as eng:
            eng.set_X(X); eng.set_pathways(packed); eng.set_UV(U, V); eng.set_active(active)
            eng.step_async(3, 2.0, 0.4)
            eng.block_end(3, want_scores=True, prefetch=prefetch)
            U1, V1 = eng.get_UV()
            eng.set_X(X2)
            parts, _, _ = eng.step(2, 2.0, 0.4)
            runs.append((parts, U1, V1) + eng.get_UV())
    for x, y in zip(*runs):
        assert np.array_equal(x, y)
    _, U1, V1 = runs[0][:3]
    with CudaEngine(300, 300, 1200, k) as fresh:
        fresh.set_X(X2); fresh.set_pathways(packed); fresh.set_UV(U1, V1); fresh.set_active(active)
        parts, _, _ = fresh.step(2, 2.0, 0.4)
        Uf, Vf = fresh.get_UV()
    np.testing.assert_allclose(parts, runs[0][0], rtol=1e-12)
    np.testing.assert_allclose(Uf, runs[0][3], rtol=1e-12, atol=1e-14)
    np.testing.assert_allclose(Vf, runs[0][4], rtol=1e-12, atol=1e-14)


@pytest.mark.gpu
@pytest.mark.parametrize("k", [6, 12])
def test_nnls_leaves_U_and_V_unset(b200, k):
    """prmf_nnls_x uses U and V as scratch.  Until both are set again, steps fail; project_t fails until U is set; once
    both are set, the steps are those of a fresh handle."""
    from prmf_b200 import CudaEngine
    from prmf_b200._lib import PrmfLibraryError
    X, packed, U, V, active = _instance(120, 400, k, 9, seed=81)
    rng = np.random.Generator(np.random.PCG64(82))
    with CudaEngine(120, 120, 400, k) as eng:
        eng.set_X(X); eng.set_pathways(packed); eng.set_UV(U, V); eng.set_active(active)
        eng.nnls(rng.random((400, k)), transpose=True)
        with pytest.raises(PrmfLibraryError):
            eng.project_t()
        eng.set_UV(None, V)
        with pytest.raises(PrmfLibraryError):
            eng.step(1, 2.0, 0.4)
        with pytest.raises(PrmfLibraryError):
            eng.project_t()
        eng.nnls(rng.random((120, k)), transpose=False)
        eng.set_UV(U, None)
        with pytest.raises(PrmfLibraryError):
            eng.step(1, 2.0, 0.4)
        with pytest.raises(PrmfLibraryError):
            eng.project()
        eng.set_UV(U, V)
        got = eng.step(3, 2.0, 0.4)[0], eng.get_UV()
    with CudaEngine(120, 120, 400, k) as fresh:
        fresh.set_X(X); fresh.set_pathways(packed); fresh.set_UV(U, V); fresh.set_active(active)
        want = fresh.step(3, 2.0, 0.4)[0], fresh.get_UV()
    assert np.array_equal(got[0], want[0])
    assert np.array_equal(got[1][0], want[1][0]) and np.array_equal(got[1][1], want[1][1])


@pytest.mark.gpu
def test_handle_without_rows(b200):
    from prmf_b200 import CudaEngine
    n, k = 131, 6
    V = _ints(np.random.Generator(np.random.PCG64(3)), n, k)
    with CudaEngine(0, 0, n, k) as eng:
        eng.set_X(np.empty((0, n)))
        eng.set_UV(None, V)
        assert eng.project().shape == (0, k)
        B = eng.project_t()
        assert B.shape == (n, k) and np.all(B == 0.0)
        assert eng.normX_sq == 0.0
