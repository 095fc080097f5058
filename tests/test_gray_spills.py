"""Register-spill guard for the one-channel preprocessing kernels (8-bit gray input).

The fused gray edge kernel is on the hot path of every gray frame; with local-memory traffic it would lose what reading a third
of the bytes gains. This test compiles ea_preprocess.cu and ea_canny_edt.cu with the project's flags plus `-Xptxas -v` and
requires ptxas (CUDA 12.9) to report no spill stores and no spill loads for the kernels that read gray input.
"""
import tempfile
from concurrent.futures import ThreadPoolExecutor

import pytest

from test_solve_spills import _nvcc, _ptxas_report

# translation unit -> mangled-name fragments of the one-channel kernels (every instantiation must be spill-free)
KERNELS = {
    "ea_preprocess.cu": ["k_edge_mask2_grayItLi128ELb1E", "k_edge_mask2_grayItLi128ELb0E", "k_edge_mask2_grayIfLi128ELb1E",
                         "k_edge_mask2_grayItLi64ELb1E", "k_edge_mask2_grayIfLi64ELb0E", "k_edge_maskItLi1E", "k_edge_maskIfLi1E",
                         "k_pyr_downItLi1E", "k_pyr_down4ItLi1E", "k_pyr_down4IfLi1E"],
    "ea_canny_edt.cu": ["k_box_grayILi1E", "k_canny_gradILi1E"],
}


def test_gray_kernels_do_not_spill():
    nvcc = _nvcc()
    if nvcc is None:
        pytest.skip("nvcc not found")
    with tempfile.TemporaryDirectory() as tmp, ThreadPoolExecutor(len(KERNELS)) as ex:
        reports = dict(zip(KERNELS, ex.map(lambda s: _ptxas_report(nvcc, s, tmp), KERNELS)))
    for src, frags in KERNELS.items():
        for frag in frags:
            hits = [r for r in reports[src] if frag in r[0]]
            assert hits, "%s: ptxas reported no function matching %s" % (src, frag)
            for name, st, ld in hits:
                assert st == 0 and ld == 0, "%s: %s spills %d B stored / %d B loaded" % (src, name, st, ld)
