"""Register-spill guard for the kernels that read camera / decoder frames in place (NV12, YUYV, UYVY, pitched gray).

Every luma layout of the fused gray edge kernel (planar, YUYV, UYVY) is a hot path for its input, and the byte kernels that take
a row pitch at run time serve the Canny, odd-width and misaligned inputs.  This test compiles ea_preprocess.cu and
ea_canny_edt.cu with the project's flags plus `-Xptxas -v` and requires ptxas (CUDA 12.9) to report no spill stores and no
spill loads for each of them.
"""
import itertools
import tempfile
from concurrent.futures import ThreadPoolExecutor

import pytest

from test_solve_spills import _nvcc, _ptxas_report

# k_edge_mask2_gray<D, TW, REF, LUMA>: depth u16 / f32, 128- / 64-wide tiles, with / without the reference plane, planar / YUYV / UYVY
EDGE2 = ["k_edge_mask2_grayI%sLi%dELb%dELi%dE" % c for c in itertools.product("tf", (128, 64), (0, 1), (0, 1, 2))]
KERNELS = {
    "ea_preprocess.cu": EDGE2 + ["k_edge_maskItLi1E", "k_edge_maskIfLi1E", "k_pyr_downItLi1E", "k_pyr_downIfLi1E",
                                 "k_pyr_down4ItLi1E", "k_pyr_down4IfLi1E"],
    "ea_canny_edt.cu": ["k_box_grayILi1E", "k_canny_gradILi1E"],
}


def test_luma_layout_kernels_do_not_spill():
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
