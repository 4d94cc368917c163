"""Static checks of the shipped SASS (no GPU needed): the hot kernels take the hardware paths DESIGN.md claims, and the
main loop of the persistent step kernel -- which lives at the register limit of a 10-warp CTA -- is free of spills and
register-move storms (both have happened when tail code grew: the cost was 25-50 % of the stream rate)."""
import os
import re
import shutil
import subprocess

import pytest

from conftest import ROOT
from test_xstream_exact import fg_kt

LIB = os.path.join(ROOT, "prmf_b200", "libprmf_b200.so")


def _sass_by_function():
    exe = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(exe) or not os.path.exists(LIB):
        pytest.skip("cuobjdump or the built library is not available")
    out = subprocess.run([exe, "-sass", LIB], capture_output=True, text=True, check=True).stdout
    funcs, cur = {}, None
    for line in out.split("\n"):
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = m.group(1)
            funcs[cur] = []
            continue
        m = re.match(r"\s*/\*[0-9a-f]+\*/\s+(?:@!?U?P\d+\s+)?([A-Z][A-Z0-9_.]*)", line)
        if cur and m:
            funcs[cur].append(m.group(1))
    return funcs


def _longest_dfma_region(ops, gap=30):
    """[start, end) of the longest stretch in which DFMAs are never more than `gap` instructions apart."""
    idx = [i for i, op in enumerate(ops) if op.startswith("DFMA")]
    best, start, prev = (0, 0), idx[0], idx[0]
    for i in idx[1:]:
        if i - prev > gap:
            if prev - start > best[1] - best[0]:
                best = (start, prev)
            start = i
        prev = i
    if prev - start > best[1] - best[0]:
        best = (start, prev)
    return best


def test_hot_kernels_use_the_claimed_hardware_paths():
    funcs = _sass_by_function()

    def ops_of(substr):
        names = [n for n in funcs if substr in n]
        assert names, "no kernel matching %s in the library" % substr
        return [op for n in names for op in funcs[n]]

    stream = ops_of("skinny_tma_kernelILi10ELi8ELi1E")
    assert any(op.startswith("UBLKCP") for op in stream) and any(op.startswith("SYNCS") for op in stream)   # TMA bulk + mbarrier
    assert sum(op.startswith("DFMA") for op in stream) >= 320
    block = ops_of("block_kernelILi10E")
    assert any(op.startswith("UBLKCP") for op in block) and any(op.startswith("SYNCS") for op in block)
    tc = ops_of("tc_rowdot_kernel")
    for needle in ("UTMALDG", "UTCHMMA", "LDTM", "UTCBAR"):                 # tensor-map TMA, tcgen05.mma, tcgen05.ld, commit
        assert any(op.startswith(needle) for op in tc), needle


def test_stream_kernel_main_loops_are_clean():
    funcs = _sass_by_function()
    for k in (6, 10):
      for pattern in ("block_kernelILi%dE" % k, "skinny_tma_kernelILi%dELi8ELi1E" % k, "skinny_tma_kernelILi%dELi8ELi2E" % k):
        name = [n for n in funcs if pattern in n][0]
        ops = funcs[name]
        a, b = _longest_dfma_region(ops)
        loop = ops[a:b + 1]
        n_dfma = sum(op.startswith("DFMA") for op in loop)
        assert n_dfma >= 8 * 4 * k, pattern                                 # the 8-row stage, 4 columns per thread
        assert not any(op.startswith(("LDL", "STL")) for op in loop), "spills inside the X-stream main loop of %s" % pattern
        moves = sum(op.startswith(("IMAD.MOV", "MOV")) for op in loop)
        assert moves <= n_dfma // 8, "register-move storm inside the main loop of %s: %d moves for %d DFMA" % (pattern, moves, n_dfma)
        assert sum(op.startswith("LDS.128") for op in loop) >= 8 * (2 + (k // 2 if k % 2 == 0 else 0)) - 16, pattern


def _instantiations(funcs, kernel):
    """The template arguments of every instantiation of the three-argument kernel template `kernel` in the library."""
    found = (re.search(kernel + r"ILi(\d+)ELi(\d+)ELi(\d+)E", n) for n in funcs)
    return {tuple(int(v) for v in m.groups()) for m in found if m}


def test_stream_kernel_instantiations_are_the_reachable_set():
    """The library holds the fp64 X-stream kernels the launch planner can select, and no others: skinny_tma_kernel at
    k = 1..10 with every fused tail (EPI 0..3), skinny_tma_gen_kernel at every (KT, FG) that k = 11..128 reaches."""
    funcs = _sass_by_function()
    assert _instantiations(funcs, "skinny_tma_kernel") == {(k, 8, epi) for k in range(1, 11) for epi in range(4)}
    assert _instantiations(funcs, "skinny_tma_gen_kernel") == {(kt, fg, 8) for fg, kt in (fg_kt(k) for k in range(11, 129))}
