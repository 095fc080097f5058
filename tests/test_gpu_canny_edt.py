"""Canny hysteresis and the exact Euclidean DT (ea_canny_edt.cu) against the oracle, bit for bit: edge masks, reference point
lists (u, v, depth, order) and distance transforms.

The bundled frames are noisy natural images whose weak edges all lie a few pixels from a strong one.  What hysteresis is for --
a long chain of weak pixels seeded from far away -- is tested on a serpentine band whose few strong pixels are near one end, so
that the farthest edge pixel is tens of thousands of 8-connected steps from the nearest strong pixel.  The exact DT is tested on
sculpted edge maps: none, a few columns (most columns have no edge pixel), all, the corners, and frames up to 3840x2160, where
the largest squared distance exceeds 2^24 and rounds when converted to float.

The CPU tests at the top run without a GPU: they keep the serpentine a long-chain test and pin the fast exact-DT reference used
for the large frames to the oracle.
"""
from collections import deque

import numpy as np
import pytest

gpu = pytest.mark.gpu

EDT_NONE = 65536.0          # OpenCV's value of every pixel when the image has no zero pixel


# ------------------------------------------------------------------------------------------------------------ fixtures
def serpentine(w, h, ramp, band_value=140, seed_value=100, period=8, band=4, margin=4):
    """A gray image with a 4-px band folded into vertical teeth of 8-px period that span the height, joined alternately at the
    bottom and the top.  The background is seed_value under the first 10 columns and ramps from ramp[0] to ramp[1] after
    them, so the band's contrast -- and with it the Canny magnitude -- is highest at the left end: strong edge pixels are few, and
    hysteresis has to carry them along the whole band."""
    m = np.zeros((h, w), bool)
    xs = list(range(margin, w - margin - band, period))
    for j, x in enumerate(xs):
        m[margin:h - margin, x:x + band] = True
        if j + 1 < len(xs):
            y = (h - margin - band) if j % 2 == 0 else margin
            m[y:y + band, x:xs[j + 1] + band] = True
    x = np.arange(w)
    bg = np.where(x < 10, seed_value, np.round(ramp[0] + (ramp[1] - ramp[0]) * x / w)).astype(np.uint8)
    g = np.broadcast_to(bg, (h, w)).copy()
    g[m] = band_value
    return g


# name -> (edge detector, low, high, L2, background ramp); tuned with the oracle so that the chains are long (see
# test_serpentine_is_a_long_chain_test)
LONG_CHAINS = {
    "gray-l1": (1, 30.0, 90.0, 0, (108, 126)),        # box blur -> gray -> Canny, the standalone variant's thresholds
    "color-l1": (2, 50.0, 150.0, 0, (108, 126)),
    "color-l2": (2, 40.0, 100.0, 1, (118, 128)),
}


def rep3(gray):
    return np.ascontiguousarray(np.repeat(np.asarray(gray, np.uint8)[..., None], 3, -1))


def to_gray(bgr):
    """OpenCV's 8-bit RGB2GRAY on BGR data."""
    b = np.asarray(bgr, np.int64)
    return ((b[..., 0] * 9798 + b[..., 1] * 19235 + b[..., 2] * 3735 + 16384) >> 15).astype(np.uint8)


def tile_to(a, w, h):
    """Frames [n][h0][w0](...) cut or tiled to w x h."""
    reps = (-(-h // a.shape[1]), -(-w // a.shape[2])) + (1,) * (a.ndim - 3)
    return np.ascontiguousarray(np.tile(a, (1,) + reps)[:, :h, :w])


def oracle_edges(O, img, detector, low, high, l2):
    """Boolean edge map of the Canny pipeline `detector` on one BGR (h, w, 3) or gray (h, w) image."""
    bgr = img if img.ndim == 3 else rep3(img)
    src = O.rgb2gray(O.box3(bgr)) if detector == 1 else bgr
    return O.canny(src, low, high, l2=bool(l2)) > 0


def edt_ref(inv):
    """Exact Euclidean DT of a u8 map (0 == feature) with the oracle's rounding -- the exact integer squared distance, converted
    to float32, then sqrtf -- and OpenCV's 65536 where the map has no zero.  O(pixels), for frames where oracle.exact_edt
    (O(w^2 h)) is too slow."""
    from scipy.ndimage import distance_transform_edt
    z = np.asarray(inv) == 0
    if not z.any():
        return np.full(z.shape, EDT_NONE, np.float32)
    d = distance_transform_edt(~z)
    return np.sqrt(np.rint(d * d).astype(np.float32))


def expected_dt(O, edges, dt_kind, norm):
    inv = np.where(edges, 0, 255).astype(np.uint8)
    d = edt_ref(inv) if dt_kind == 1 else O.chamfer3_dt(inv)
    return d if norm == 0 else O.normalize_minmax(d, 0, 1.0 if norm == 1 else 255.0)


def expected_points(edges, depth, zero_to_one, depth_one):
    """get_aX's list: edge pixels with depth (or every edge pixel, depth 0 kept at Z = 1) in row-major order."""
    keep = edges if zero_to_one else edges & (depth > 0)
    vs, us = np.nonzero(keep)
    z = depth[vs, us].astype(np.float32)
    if zero_to_one:
        z[z == 0] = depth_one
    return np.stack([us, vs, z, np.ones_like(z)], 1).astype(np.float32)


def geodesic(cand, strong):
    """Largest 8-connected step count from the strong set to a pixel of cand reachable from it, and the reached set."""
    h, w = cand.shape
    dist = np.full((h, w), -1, np.int64)
    q = deque()
    for y, x in zip(*np.nonzero(strong)):
        dist[y, x] = 0
        q.append((y, x))
    while q:
        y, x = q.popleft()
        d = dist[y, x] + 1
        for yy in (y - 1, y, y + 1):
            for xx in (x - 1, x, x + 1):
                if 0 <= yy < h and 0 <= xx < w and cand[yy, xx] and dist[yy, xx] < 0:
                    dist[yy, xx] = d
                    q.append((yy, xx))
    return int(dist.max()), dist >= 0


# ---------------------------------------------------------------------------------------------- CPU preconditions
@pytest.mark.parametrize("geom", [(640, 512), (640, 480)])
@pytest.mark.parametrize("path", sorted(LONG_CHAINS))
def test_serpentine_is_a_long_chain_test(oracle, path, geom):
    """From the oracle alone: every pixel of the final edge map is reached from the strong pixels, and the farthest one is at
    least 20 000 8-connected steps away from them.  On the L1 paths every candidate (NMS maximum above low) is
    reached, so the final map is the whole band's edge."""
    O = oracle
    w, h = geom
    det, low, high, l2, ramp = LONG_CHAINS[path]
    img = serpentine(w, h, ramp)
    cand = oracle_edges(O, img, det, low, low, l2)          # high == low: every NMS maximum above low is strong
    strong = oracle_edges(O, img, det, high, high, l2)
    final = oracle_edges(O, img, det, low, high, l2)
    far, reached = geodesic(cand, strong)
    np.testing.assert_array_equal(final, reached)
    assert far >= 20000, far
    if not l2:
        np.testing.assert_array_equal(final, cand)
        assert final.sum() > 60000


def _edt_cases(rng):
    yield "random", [(rng.random((h, w)) > p).astype(np.uint8) * 255
                     for (w, h, p) in ((1, 1, 0.5), (7, 3, 0.3), (64, 48, 0.02), (256, 17, 0.001), (131, 200, 0.0005), (256, 256, 0.9))]
    yield "no edge", [np.full((48, 64), 255, np.uint8), np.full((1, 1), 255, np.uint8)]
    cols = np.full((48, 64), 255, np.uint8); cols[[3, 30], 5] = 0; cols[47, 60] = 0
    yield "few columns", [cols]
    yield "all edges", [np.zeros((48, 64), np.uint8)]
    corners = []
    for (y, x) in ((0, 0), (0, 63), (47, 0), (47, 63)):
        c = np.full((48, 64), 255, np.uint8); c[y, x] = 0; corners.append(c)
    c = np.full((48, 64), 255, np.uint8); c[[0, 0, 47, 47], [0, 63, 0, 63]] = 0
    yield "corners", corners + [c]


def test_fast_edt_reference_equals_oracle(oracle):
    """edt_ref (scipy, O(pixels)) == oracle.exact_edt (OpenCV's trueDistTrans restated, O(w^2 h)) bit for bit."""
    rng = np.random.default_rng(7)
    for name, maps in _edt_cases(rng):
        for m in maps:
            np.testing.assert_array_equal(edt_ref(m), oracle.exact_edt(m), err_msg="%s %s" % (name, m.shape))


def test_fast_edt_reference_rounds_above_2_24():
    """Above 2^24 the integer squared distance is rounded to float32 before the square root, as the kernel and the oracle do."""
    m = np.full((2160, 3840), 255, np.uint8); m[0, 0] = 0
    d = edt_ref(m)
    d2 = 3839 ** 2 + 2158 ** 2
    assert d2 > 1 << 24 and float(np.float32(d2)) != d2
    assert d[2158, 3839] == np.sqrt(np.float32(d2))
    assert d[0, 1] == 1.0 and d[1, 1] == np.float32(np.sqrt(2.0))


# ------------------------------------------------------------------------------------------------------- GPU tests
@pytest.fixture(scope="module")
def ea():
    import edge_alignment_b200 as ea
    return ea


@pytest.fixture(scope="module")
def ctx(ea):
    c = ea.Context(0)
    yield c
    c.close()


def _fp(ea, w, h, **kw):
    return ea.frame_params(width=w, height=h, fx=525.0 * w / 640, fy=525.0 * w / 640, cx=(w - 1) / 2, cy=(h - 1) / 2,
                           max_points=w * h, **kw)


def _half(img):
    from oracle import oracle as O
    bgr = img if img.ndim == 3 else rep3(img)
    return O.half_linear(bgr) if img.ndim == 3 else O.half_linear(bgr)[..., 0].copy()


def _half_depth(d):
    from oracle import oracle as O
    return O.half_nearest(d) if d.dtype == np.uint16 else np.ascontiguousarray(d[::2, ::2])


def check_frames(ea, O, fs, fp, slots, imgs, depths, roles, what=""):
    """Every frame, every level: edge mask, point list (if REF) and DT (if NOW) against the oracle.  imgs are BGR or gray as fed."""
    det, low, high, l2 = fp.edge_detector, fp.canny_low, fp.canny_high, fp.canny_l2
    depth_one = 1.0 if fp.depth_type == ea.DEPTH_F32 else fp.depth_scale
    for i, (slot, img) in enumerate(zip(slots, imgs)):
        dep = depths[i] if depths is not None else None
        for l in range(fp.n_levels):
            where = "%s frame %d slot %d level %d" % (what, i, slot, l)
            edges = oracle_edges(O, img, det, low, high, l2)
            got = fs.edge_mask(int(slot), l) == 0
            bad = int((got != edges).sum())
            assert bad == 0, "%s: %d of %d edge pixels differ (%d missing, %d extra)" % (
                where, bad, int(edges.sum()), int((edges & ~got).sum()), int((got & ~edges).sum()))
            if roles & ea.ROLE_REF:
                np.testing.assert_array_equal(fs.points(int(slot), l), expected_points(edges, dep, fp.zero_depth_to_one, depth_one),
                                              err_msg=where)
            if roles & ea.ROLE_NOW:
                np.testing.assert_array_equal(fs.dt(int(slot), l), expected_dt(O, edges, fp.dt_kind, fp.dt_normalize), err_msg=where)
            if l + 1 < fp.n_levels:
                img = _half(img)
                dep = _half_depth(dep) if dep is not None else None


def _preprocess(fs, entry, slots, imgs, depth, roles):
    if entry == "gray":
        fs.preprocess_gray_host(slots, np.stack(imgs), depth, roles)
    else:
        fs.preprocess_host(slots, np.stack([im if im.ndim == 3 else rep3(im) for im in imgs]), depth, roles)


# ---------------------------------------------------------------------------------------------- a. long edge chains
@gpu
@pytest.mark.parametrize("dt_kind", ["exact", "chamfer"])
@pytest.mark.parametrize("entry", ["bgr", "gray"])
@pytest.mark.parametrize("geom", ["640x512", "640x480"])
@pytest.mark.parametrize("path", sorted(LONG_CHAINS))
def test_long_chains_match_oracle(ea, ctx, frames, oracle, path, geom, entry, dt_kind):
    """Serpentine frames (seeded at the left, and mirrored so that the flood runs the other way through memory) between bundled
    frames in one batch, scrambled slots, two pyramid levels (level 1 of 640x512 is 320x256): every frame's edges must be the
    oracle's 8-connected closure of its strong pixels, and neither a slow flood nor its scratch may leak into another frame."""
    w, h = (int(v) for v in geom.split("x"))
    det, low, high, l2, ramp = LONG_CHAINS[path]
    s = serpentine(w, h, ramp)
    bundled = tile_to(frames["bgr"][[0, 2, 4]], w, h)
    if entry == "gray":
        bundled = to_gray(bundled)
    else:
        s = rep3(s)
    imgs = [s, bundled[0], np.ascontiguousarray(s[:, ::-1]), bundled[1], np.ascontiguousarray(s[::-1]), bundled[2]]
    n = len(imgs)
    rng = np.random.default_rng(w + h + det)
    d16 = tile_to(frames["depth"][:1], w, h)[0]
    depth = np.stack([np.roll(d16, 9 * i, axis=0) for i in range(n)])
    depth[::2] *= (rng.random((n - n // 2, h, w)) > 0.2).astype(np.uint16)          # serpentine frames: holes in the depth
    slots = rng.permutation(n + 2)[:n].astype(np.int32)
    fp = _fp(ea, w, h, n_levels=2, edge_detector=det, canny_low=low, canny_high=high, canny_l2=l2,
             dt_kind=ea.DT_EXACT if dt_kind == "exact" else ea.DT_CHAMFER3, dt_normalize=ea.NORM_255 if dt_kind == "exact" else ea.NORM_01)
    fs = ea.FrameSet(ctx, fp, n + 2)
    try:
        _preprocess(fs, entry, slots, imgs, depth, ea.ROLE_BOTH)
        check_frames(ea, oracle, fs, fp, slots, imgs, depth, ea.ROLE_BOTH, path)
    finally:
        fs.close()


# ------------------------------------------------------------------------------------ b. threshold and NMS conventions
def convention_images(w=64, h=48):
    """BGR frames with known Sobel magnitudes: steps of several heights in the four NMS sectors, 1- and 2-px ridges and
    valleys (horizontal, vertical, both diagonals: the > / >= asymmetry of the comparisons and the sign sg of the diagonal
    sector decide which pixel of a 2-px ridge survives), and colour frames whose channels tie in magnitude with opposite
    gradient signs (first channel wins) or differ only in one channel."""
    yy, xx = np.mgrid[0:h, 0:w]
    imgs = []
    for d, cond in ((37, xx >= 20), (53, yy >= 17), (61, xx + yy >= 40), (29, xx - yy >= 10), (90, (xx - 32) ** 2 + (yy - 24) ** 2 < 200)):
        g = np.full((h, w), 60, np.int64); g[cond] += d; imgs.append(rep3(g))
    for width in (1, 2):
        for k, t in enumerate((yy - 20, xx - 30, xx - yy - 8, xx + yy - 50)):
            g = np.full((h, w), 110, np.int64); g[(t >= 0) & (t < width)] += 45 if k % 2 == 0 else -45; imgs.append(rep3(g))
    tie = np.full((h, w, 3), 100, np.int64)
    tie[..., 0][xx + yy >= 40] += 40; tie[..., 1][xx + yy >= 40] -= 40                # equal magnitudes, opposite signs
    tie[..., 2][(xx - yy >= 5) & (xx - yy < 7)] += 70                                # a 2-px diagonal ridge in one channel only
    imgs.append(tie)
    one = np.full((h, w, 3), 90, np.int64); one[..., 1][10:30, 12] = 160; one[..., 0][30, 5:60] = 20
    imgs.append(one)
    return [np.clip(im, 0, 255).astype(np.uint8) for im in imgs]


def sobel_mag(O, img, detector, l2):
    """The magnitude plane the Canny of `detector` compares with its thresholds (channel of largest magnitude)."""
    src = O.rgb2gray(O.box3(img)) if detector == 1 else img
    a = np.asarray(src, np.int64)
    a = a[..., None] if a.ndim == 2 else a
    p = np.pad(a, ((1, 1), (1, 1), (0, 0)), mode="edge")
    dx = (p[:-2, 2:] + 2 * p[1:-1, 2:] + p[2:, 2:]) - (p[:-2, :-2] + 2 * p[1:-1, :-2] + p[2:, :-2])
    dy = (p[2:, :-2] + 2 * p[2:, 1:-1] + p[2:, 2:]) - (p[:-2, :-2] + 2 * p[:-2, 1:-1] + p[:-2, 2:])
    return (dx * dx + dy * dy if l2 else np.abs(dx) + np.abs(dy)).max(-1)


def threshold_cases(mags, l2):
    """(low, high) pairs pinning `m > low` and `m > high` at present magnitudes m and m +- 1, fractional thresholds (floored),
    swapped and equal thresholds, and for L2 thresholds above sqrt of the largest magnitude and above 32767 (clamped)."""
    u = np.unique(mags[mags > 0])
    lo, mid, top = int(u[len(u) // 4]), int(u[len(u) // 2]), int(u[-1])
    t = (lambda k: float(np.sqrt(k + 0.5))) if l2 else float      # threshold whose floored (squared) value is k
    cases = [(t(lo + d), t(mid)) for d in (-1, 0, 1)] + [(t(lo), t(mid + d)) for d in (-1, 0, 1)]
    cases += [(t(lo), t(top + d)) for d in (-1, 0)] + [(t(mid), t(lo)), (t(mid), t(mid)), (t(lo - 1), t(lo - 1))]
    if l2:
        cases += [(np.sqrt(lo) + 0.25, np.sqrt(mid) + 0.75), (1.0, np.sqrt(top) + 1.0), (3.0, 50000.0), (40000.0, 60000.0)]
    else:
        cases += [(lo + 0.5, mid + 0.999), (lo - 0.25, mid - 0.5)]
    return cases


@gpu
@pytest.mark.parametrize("l2", [0, 1])
@pytest.mark.parametrize("det", [1, 2])
def test_threshold_and_nms_conventions(ea, ctx, oracle, det, l2):
    O = oracle
    bgr = convention_images()
    w, h = 64, 48
    mags = np.stack([sobel_mag(O, im, det, l2) for im in bgr])
    for low, high in threshold_cases(mags, l2):
        fp = _fp(ea, w, h, edge_detector=det, canny_low=low, canny_high=high, canny_l2=l2, dt_kind=ea.DT_EXACT, dt_normalize=ea.NORM_NONE)
        for entry in ("bgr", "gray"):
            imgs = bgr if entry == "bgr" else [to_gray(im) for im in bgr]
            slots = np.arange(len(imgs))[::-1].copy()
            fs = ea.FrameSet(ctx, fp, len(imgs))
            try:
                _preprocess(fs, entry, slots, imgs, None, ea.ROLE_NOW)
                check_frames(ea, O, fs, fp, slots, imgs, None, ea.ROLE_NOW, "%s thresholds %r %r" % (entry, low, high))
            finally:
                fs.close()


# ----------------------------------------------------------------------------------------------------- c. shape sweep
# (w, h, levels): runs of pixels per thread of a 1024-thread CTA shorter than a row (31, 33, 255, 257, 641), half a row
# (1000x512), longer than a row (100x1100), and 8x8, where most threads of such a CTA would own no pixel
SHAPES = [(8, 8, 1), (31, 40, 1), (33, 62, 1), (100, 1100, 3), (255, 24, 1), (257, 30, 1), (641, 20, 1), (1000, 512, 3)]


@gpu
@pytest.mark.parametrize("shape", SHAPES, ids=["%dx%d" % s[:2] for s in SHAPES])
def test_canny_shapes(ea, ctx, oracle, shape):
    w, h, levels = shape
    k = SHAPES.index(shape)
    rng = np.random.default_rng(100 + k)
    n = 3
    blocks = rng.integers(0, 4, (n, h // 3 + 1, w // 3 + 1, 3)) * 70 + rng.integers(0, 12, (n, h // 3 + 1, w // 3 + 1, 3))
    bgr = np.ascontiguousarray(np.repeat(np.repeat(blocks, 3, 1), 3, 2)[:, :h, :w].astype(np.uint8))
    bgr[1] = rep3(to_gray(bgr[1]))                          # a gray-valued frame too
    d16 = (rng.integers(0, 3, (n, h, w)) * 900).astype(np.uint16)
    f32 = k % 2 == 1
    depth = (d16.astype(np.float32) / 5000.0) if f32 else d16
    det = 1 + k % 2
    fp = _fp(ea, w, h, n_levels=levels, edge_detector=det, canny_low=150.0 if det == 2 else 30.0, canny_high=100.0 if det == 2 else 90.0,
             canny_l2=(k // 2) % 2, dt_kind=ea.DT_EXACT if k % 3 != 2 else ea.DT_CHAMFER3, dt_normalize=k % 3,
             depth_type=ea.DEPTH_F32 if f32 else ea.DEPTH_U16, zero_depth_to_one=int(k % 4 == 3 or k == 0))
    slots = rng.permutation(n + 1)[:n].astype(np.int32)
    fs = ea.FrameSet(ctx, fp, n + 1)
    try:
        fs.preprocess_host(slots, bgr, depth, ea.ROLE_BOTH)
        check_frames(ea, oracle, fs, fp, slots, list(bgr), depth, ea.ROLE_BOTH, "%dx%d" % (w, h))
    finally:
        fs.close()


# ------------------------------------------------------------------------------------------------ d. exact EDT edges
def edt_frameset(ea, ctx, w, h, n, n_levels=1, norm=0):
    """A frame set whose edge map is exactly the now-mask: the Laplacian detector with threshold -1 marks every pixel, and
    preprocess_now_masked keeps the pixels where mask > 1."""
    fp = _fp(ea, w, h, n_levels=n_levels, grad_threshold=-1, use_median=0, dt_kind=ea.DT_EXACT, dt_normalize=norm)
    return ea.FrameSet(ctx, fp, n)


def run_edt(ea, fs, masks, slots, ref):
    n_levels = fs.params.n_levels
    w, h = fs.params.width, fs.params.height
    fs.preprocess_now_masked(slots, np.zeros((len(masks), h, w, 3), np.uint8), np.stack(masks))
    for i, (slot, m) in enumerate(zip(slots, masks)):
        for l in range(n_levels):
            edges = m[::1 << l, ::1 << l] > 1
            where = "frame %d level %d" % (i, l)
            np.testing.assert_array_equal(fs.edge_mask(int(slot), l) == 0, edges, err_msg=where)
            np.testing.assert_array_equal(fs.dt(int(slot), l), ref(edges), err_msg=where)


@gpu
@pytest.mark.parametrize("norm", [0, 1, 2])
def test_exact_edt_sculpted_edges(ea, ctx, oracle, norm):
    """No edge pixel (65536 everywhere; normalised over a zero range: 0), edges in three columns only, every pixel an edge, one
    corner pixel per frame and all four corners; two levels (level 1 samples the mask at even pixels), scrambled slots."""
    O = oracle
    w, h = 96, 64
    masks = [np.zeros((h, w), np.uint8)]
    m = np.zeros((h, w), np.uint8); m[[6, 40], 4] = 255; m[[0, 63], 50] = 7; m[22, 94] = 2; masks.append(m)
    masks.append(np.full((h, w), 200, np.uint8))
    for (y, x) in ((0, 0), (0, w - 2), (h - 2, 0), (h - 1, w - 1)):
        m = np.zeros((h, w), np.uint8); m[y, x] = 255; masks.append(m)
    m = np.zeros((h, w), np.uint8); m[[0, 0, h - 2, h - 2], [0, w - 2, 0, w - 2]] = 9; masks.append(m)
    slots = np.random.default_rng(norm).permutation(len(masks)).astype(np.int32)

    def ref(edges):
        d = O.exact_edt(np.where(edges, 0, 255).astype(np.uint8))
        return d if norm == 0 else O.normalize_minmax(d, 0, 1.0 if norm == 1 else 255.0)

    fs = edt_frameset(ea, ctx, w, h, len(masks), n_levels=2, norm=norm)
    try:
        run_edt(ea, fs, masks, slots, ref)
        if norm == 0:
            assert np.all(fs.dt(int(slots[0])) == EDT_NONE)
        else:
            assert np.all(fs.dt(int(slots[0])) == 0) and np.all(fs.dt(int(slots[2])) == 0)
    finally:
        fs.close()


@gpu
@pytest.mark.parametrize("geom", ["1280x720", "1920x1080"])
def test_exact_edt_large_frames_vs_oracle(ea, ctx, oracle, geom):
    """One frame of sparse random edges and empty bands (the row search runs far before it can stop) against oracle.exact_edt."""
    w, h = (int(v) for v in geom.split("x"))
    rng = np.random.default_rng(w)
    m = ((rng.random((h, w)) < 2e-4) * 255).astype(np.uint8)
    m[:, w // 3: w // 2] = 0; m[h // 4: h // 2] = 0
    fs = edt_frameset(ea, ctx, w, h, 2)
    try:
        run_edt(ea, fs, [m], [1], lambda e: oracle.exact_edt(np.where(e, 0, 255).astype(np.uint8)))
    finally:
        fs.close()


@gpu
def test_exact_edt_4k_squared_distance_above_2_24(ea, ctx):
    """3840x2160, a single edge pixel in one corner, then in the opposite one: squared distances up to 19.4 M round when
    converted to float before the square root; against the scipy reference pinned to the oracle above."""
    w, h = 3840, 2160
    masks = [np.zeros((h, w), np.uint8), np.zeros((h, w), np.uint8)]
    masks[0][0, 0] = 255; masks[1][h - 1, w - 1] = 255
    fs = edt_frameset(ea, ctx, w, h, 2)
    try:
        run_edt(ea, fs, masks, [1, 0], lambda e: edt_ref(np.where(e, 0, 255).astype(np.uint8)))
    finally:
        fs.close()
