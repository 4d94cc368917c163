"""N > 1 path: rows of X and U sharded over ranks, partial X^T U / U^T U summed over ranks.

CPU (gloo, world_size 2, numpy stand-in engine): the host logic -- sharding, identical RNG streams and
decisions on every rank, gather of U -- reproduces the reference fixture.
GPU (nccl, needs >= 2 devices): the CUDA engines with the in-library NCCL all-reduce do the same."""
import json
import os
import socket
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT, load_golden

WORKER = os.path.join(ROOT, "tests", "mp_worker.py")


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _run(case, tmp_path, world, mode, extra_env=None):
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world),
           "--master-addr", "127.0.0.1", "--master-port", str(_free_port()), WORKER, case, str(tmp_path), mode]
    env = dict(os.environ, OMP_NUM_THREADS="2", OPENBLAS_NUM_THREADS="2")
    env.update(extra_env or {})
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=900, env=env)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    return [np.load(os.path.join(tmp_path, "rank%d.npz" % r)) for r in range(world)]


def _check(case, outs, rtol_obj, rtol_uv):
    g = load_golden(case)
    meta = g["meta"]
    for z in outs:
        assert z["sampled"].tolist() == meta["sampled"]
        assert z["obj_parts"].shape == g["obj_parts"].shape
        np.testing.assert_allclose(z["obj_parts"], g["obj_parts"], rtol=rtol_obj, atol=1e-11)
        np.testing.assert_allclose(z["U"], g["U_final"], rtol=rtol_uv, atol=1e-10)
        np.testing.assert_allclose(z["V"], g["V_final"], rtol=rtol_uv, atol=1e-10)
        fm = {k: [p for p, _ in v] for k, v in meta["final_map"].items()}
        assert json.loads(str(z["fmap"])) == fm
    for z in outs[1:]:                      # every rank returns the same full result, bit for bit
        np.testing.assert_array_equal(z["U"], outs[0]["U"])
        np.testing.assert_array_equal(z["V"], outs[0]["V"])


@pytest.mark.parametrize("case", ["small_tradeoff", "test2_raw"])
def test_two_ranks_gloo_host_logic(case, tmp_path):
    outs = _run(case, tmp_path, 2, "cpu")
    _check(case, outs, rtol_obj=1e-9, rtol_uv=1e-6)


def test_three_ranks_gloo_ragged_shards(tmp_path):
    """40 rows over 3 ranks -> 14 + 14 + 12."""
    outs = _run("small_tradeoff", tmp_path, 3, "cpu")
    _check("small_tradeoff", outs, rtol_obj=1e-9, rtol_uv=1e-6)


def test_row_block_partition():
    from prmf_b200.dist import row_block
    for m, w in [(37032, 8), (10, 3), (5, 8), (100, 1), (0, 2)]:
        blocks = [row_block(m, w, r) for r in range(w)]
        assert blocks[0][0] == 0 and blocks[-1][1] == m
        for (a, b), (c, d) in zip(blocks[:-1], blocks[1:]):
            assert b == c and a <= b and c <= d


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["small_planted", "test1_norm"])
def test_two_gpus_nccl(case, tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs (run with gpurun --gpus 2); the one-device variant is test_two_ranks_on_one_gpu")
    outs = _run(case, tmp_path, 2, "gpu")
    _check(case, outs, rtol_obj=1e-9, rtol_uv=1e-6)


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["small_planted", "test1_norm"])
def test_two_ranks_on_one_gpu(case, tmp_path):
    """The sharded path on a box with ONE GPU: two processes share device 0, no NCCL (it refuses two ranks per device);
    the per-step exchange inside the persistent step kernel and the set-up reductions go through CUDA-IPC peer buffers.
    The two resident kernels wait for each other while the driver time-slices them, so every exchange costs a time
    slice -- slow, but it is the same code as on NVLink, checked against the reference fixtures."""
    cmd_env = {"PRMF_NCCL": "0", "PRMF_SPIN_TIMEOUT_MS": "4000", "CUDA_VISIBLE_DEVICES": os.environ.get("CUDA_VISIBLE_DEVICES", "0").split(",")[0]}
    try:
        outs = _run(case, tmp_path, 2, "gpu", cmd_env)
    except AssertionError as exc:
        # whether two processes can share this GPU this way is a property of the box (time slicing that interleaves two
        # resident kernels, CUDA IPC between them); the numerical checks below are not lenient
        text = str(exc)
        for marker in ("wait expired", "cudaIpc", "IPC", "peer"):
            if marker in text:
                pytest.skip("two ranks could not share this GPU (%s): %s" % (marker, text[-300:]))
        raise
    _check(case, outs, rtol_obj=1e-9, rtol_uv=1e-6)


@pytest.mark.gpu
@pytest.mark.parametrize("k,env", [
    (6, {"PRMF_P2P": "0"}),       # ncclAllReduce of the packed buffer
    (24, {}),                     # large k: tiled U / V updates, NVLink peer loads inside the tiled V update
    (24, {"PRMF_P2P": "0"}),
], ids=["6-env1", "24-env2", "24-env3"])   # fixed ids: a case keeps its id when other cases are added or removed
def test_two_gpus_match_one_gpu(k, env, tmp_path):
    """Sharded runs (all exchange flavours) against the same solve on one GPU: identical sampled pathways and
    maps, objective parts rel 1e-9, U / V rel 1e-6; all ranks bitwise equal."""
    import contextlib
    import io
    import random
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs (run with gpurun --gpus 2)")
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import mp_worker
    from prmf_b200 import nmf_pathway
    outs = _run("synth:%d" % k, tmp_path, 2, "gpu", env)
    g = mp_worker.synthetic_case(k)
    meta = g["meta"]
    np.random.seed(meta["seed"]); random.seed(meta["seed"])
    trace = {"keep_blocks": 0}
    with contextlib.redirect_stdout(io.StringIO()), contextlib.redirect_stderr(io.StringIO()):
        U, V, od = nmf_pathway(g["X"].copy(), [G.copy() for G in g["Gs"]], k_latent=k, nodelist=list(g["nodelist"]),
                               max_iter=meta["max_iter"], trace=trace)
    for z in outs:
        assert z["sampled"].tolist() == trace["sampled"]
        np.testing.assert_allclose(z["obj_parts"], np.array(trace["obj_parts"]), rtol=1e-9, atol=1e-11)
        np.testing.assert_allclose(z["U"], U, rtol=1e-6, atol=1e-10)
        np.testing.assert_allclose(z["V"], V, rtol=1e-6, atol=1e-10)
        assert json.loads(str(z["fmap"])) == {str(kk): [int(p) for p, _ in v] for kk, v in od["latent_to_pathway_data"].items()}
    np.testing.assert_array_equal(outs[1]["U"], outs[0]["U"])
    np.testing.assert_array_equal(outs[1]["V"], outs[0]["V"])
