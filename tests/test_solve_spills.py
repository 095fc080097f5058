"""Register-spill guard for the serial section between two evaluations of the persistent solve kernels.

The warp-cooperative LM step (ea_lm_advance_warp) runs in the 128-register budget of the solve kernels while the other 15
warps of the CTA wait at a barrier. Spilled to local memory, its loads miss the L1 that the evaluation sweep has just
filled with distance transform, and the step becomes several times slower than its fp64 dependency chains. This test compiles
the translation units that contain it with the project's flags plus `-Xptxas -v` and checks ptxas' spill report. The
serial state machine (ea_lm_advance, ea_lm_propose_slow) only runs on rare paths and may spill.

The limits are ptxas' figures for CUDA 12.9. The fast track's spill loads in ea_solve.cu are its pointer arguments, which
the kernel hands over in its stack frame. They are not spills of the LM state.
"""
import os
import re
import shutil
import subprocess
import tempfile
from concurrent.futures import ThreadPoolExecutor

import pytest

from conftest import ROOT

# function-name fragment -> (max spill stores, max spill loads), in bytes, per translation unit
LIMITS = {
    "ea_solve.cu": {
        "ea_lm_advance_warp": (0, 40),
        "ea_k_solve_batchILi512ELb0E": (48, 88),
        "ea_k_solve_batchILi512ELb1E": (64, 88),
    },
    "ea_shard.cu": {
        "ea_lm_advance_warp": (0, 0),
        "k_shard_solveILi512E": (52, 148),
    },
    "ea_views.cu": {
        "ea_lm_advance_warp": (0, 0),
        "k_views_solve": (0, 0),
        "k_view_eval_sums": (0, 0),
    },
}


def _nvcc():
    from edge_alignment_b200 import build
    try:
        c = build.nvcc()
    except RuntimeError:
        return None
    return c if os.path.exists(c) or shutil.which(c) else None


def _ptxas_report(nvcc, src, out_dir):
    from edge_alignment_b200 import build
    cmd = [nvcc] + build.NVCC_FLAGS + ["-Xptxas", "-v", "-c", os.path.join(build.CSRC, src),
                                       "-o", os.path.join(out_dir, src.replace(".cu", ".o"))]
    p = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert p.returncode == 0, p.stdout[-4000:]
    # every "Function properties for <name>" line is followed by its frame / spill line; a device function appears once per
    # kernel that calls it
    found = []
    name = None
    for line in p.stdout.splitlines():
        m = re.search(r"Function properties for (\S+)", line)
        if m:
            name = m.group(1)
            continue
        m = re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", line)
        if m and name:
            found.append((name, int(m.group(2)), int(m.group(3))))
            name = None
    return found


def test_lm_step_and_solve_kernels_do_not_spill_more():
    nvcc = _nvcc()
    if nvcc is None:
        pytest.skip("nvcc not found")
    with tempfile.TemporaryDirectory() as tmp, ThreadPoolExecutor(len(LIMITS)) as ex:
        reports = dict(zip(LIMITS, ex.map(lambda s: _ptxas_report(nvcc, s, tmp), LIMITS)))
    for src, limits in LIMITS.items():
        for frag, (max_st, max_ld) in limits.items():
            hits = [r for r in reports[src] if frag in r[0]]
            assert hits, "%s: ptxas reported no function matching %s" % (src, frag)
            for name, st, ld in hits:
                assert st <= max_st and ld <= max_ld, \
                    "%s: %s spills %d B stored / %d B loaded (limit %d / %d)" % (src, name, st, ld, max_st, max_ld)
