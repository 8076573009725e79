"""Oracle (our CPU restatement) against the real reference compiled from source: the reference's outputs for these
calls are stored in tests/golden/ref_outputs.npz (util.expect_ref; tests/golden/make_ref_outputs.py records them from
oracle/_ref/libmagickref.so)."""
import ctypes as C
import os

import numpy as np
import pytest

import util
from util import OUT, InOut, P, expect_ref, make_image, max_ulp, oracle


@pytest.mark.parametrize("ch", [1, 2, 3, 4])
@pytest.mark.parametrize("kind", ["noise", "alpha_blocks", "hdr"])
def test_blur_family_bit_exact(ch, kind):
    src = make_image(53, 37, ch, seed=ch * 11, kind=kind)
    o = oracle()
    for rf, of, args in (("ref_blur", o.orc_blur, (0.0, 2.0)), ("ref_blur", o.orc_blur, (0.0, 5.0)),
                         ("ref_blur", o.orc_blur, (4.0, 1.2)), ("ref_gaussian_blur", o.orc_gaussian_blur, (0.0, 1.3)),
                         ("ref_unsharp", o.orc_unsharp, (0.0, 1.5, 2.0, 0.01))):
        b = np.empty_like(src)
        assert of(P(src), P(b), 53, 37, ch, *args) == 0
        expect_ref(b, rf, src, OUT, 53, 37, ch, *args)


@pytest.mark.parametrize("ch", [1, 2, 3, 4])
@pytest.mark.parametrize("kind", ["noise", "alpha_blocks", "hdr"])
def test_sharpen_edge_bit_exact(ch, kind):
    """effect.c:3991 SharpenImage / :1520 EdgeImage: inline kernels (negative taps) + ConvolveImage."""
    src = make_image(53, 37, ch, seed=7, kind=kind)
    o = oracle()
    for rad, sig in ((0.0, 1.0), (0.0, 2.0), (2.0, 0.7), (0.0, 0.5)):
        b = np.empty_like(src)
        assert o.orc_sharpen(P(src), P(b), 53, 37, ch, rad, sig) == 0
        expect_ref(b, "ref_sharpen", src, OUT, 53, 37, ch, rad, sig)
    for rad in (0.0, 1.0, 2.0):
        b = np.empty_like(src)
        assert o.orc_edge(P(src), P(b), 53, 37, ch, rad) == 0
        expect_ref(b, "ref_edge", src, OUT, 53, 37, ch, rad)


@pytest.mark.parametrize("ch", [1, 2, 3, 4])
def test_sample_bit_exact(ch):
    """resize.c:3907 SampleImage: the double offset arithmetic picks identical source samples."""
    src = make_image(131, 77, ch, seed=9)
    for ow, oh in ((65, 38), (66, 39), (262, 154), (131, 40), (50, 77), (300, 20), (1, 1), (7, 5), (1000, 3)):
        b = np.empty((oh, ow, ch), np.float32)
        assert oracle().orc_sample(P(src), 131, 77, ch, P(b), ow, oh) == 0
        expect_ref(b, "ref_sample", src, 131, 77, ch, OUT, ow, oh, exact_bits=True)


@pytest.mark.parametrize("ch", [1, 2, 3, 4])
@pytest.mark.parametrize("kind", ["noise", "alpha_blocks", "hdr"])
def test_motion_blur_oracle_bit_exact(ch, kind):
    """effect.c:2347 MotionBlurImage -- oracle groundwork for the next hot-path row (SURVEY 8f rank 4)."""
    src = make_image(61, 47, ch, seed=13, kind=kind)
    for rad, sig, ang in ((0, 2, 0), (0, 2, 45), (0, 3, 90), (0, 1.5, -30), (0, 4, 180), (5, 2, 270), (0, 2, 123.4)):
        b = np.empty_like(src)
        assert oracle().orc_motion_blur(P(src), P(b), 61, 47, ch, rad, sig, ang) == 0
        expect_ref(b, "ref_motion_blur", src, OUT, 61, 47, ch, rad, sig, ang)


@pytest.mark.parametrize("ch", [1, 2, 3, 4])
@pytest.mark.parametrize("kind", ["noise", "alpha_blocks", "gradient"])
def test_bilateral_blur_oracle_bit_exact(ch, kind):
    """effect.c:871 BilateralBlurImage (odd windows) -- oracle groundwork for SURVEY 8f rank 4."""
    src = make_image(47, 33, ch, seed=17, kind=kind)
    for W, H, isig, ssig in ((3, 3, 10.0, 1.0), (5, 5, 20.0, 2.0), (7, 3, 8.0, 1.5), (1, 1, 5.0, 1.0), (5, 9, 30.0, 3.0)):
        b = np.empty_like(src)
        assert oracle().orc_bilateral_blur(P(src), P(b), 47, 33, ch, W, H, isig, ssig) == 0
        expect_ref(b, "ref_bilateral_blur", src, OUT, 47, 33, ch, W, H, isig, ssig)


@pytest.mark.parametrize("ch", [1, 2, 3, 4])
@pytest.mark.parametrize("kind", ["noise", "alpha_blocks", "hdr"])
def test_rotational_blur_oracle_bit_exact(ch, kind):
    """effect.c:3129 RotationalBlurImage -- oracle groundwork for SURVEY 8f rank 4."""
    src = make_image(61, 47, ch, seed=19, kind=kind)
    for ang in (5.0, 20.0, 45.0, -10.0, 90.0, 1.0):
        b = np.empty_like(src)
        assert oracle().orc_rotational_blur(P(src), P(b), 61, 47, ch, ang) == 0
        expect_ref(b, "ref_rotational_blur", src, OUT, 61, 47, ch, ang)


@pytest.mark.parametrize("ch", [1, 2, 3, 4])
@pytest.mark.parametrize("kind", ["noise", "hdr", "gradient"])
def test_statistic_oracle_bit_exact(ch, kind):
    """statistic.c:2918 StatisticImage (Gradient, Maximum, Mean, Median via the 16-bit skip list, Minimum,
    RootMeanSquare, StandardDeviation, Contrast; Mode and Nonpeak walk the same list; odd, even and 1-wide windows).  The
    posterised copy has few distinct levels, so counts tie and the median sits on the smallest / largest level."""
    src = make_image(47, 33, ch, seed=23, kind=kind)
    poster = (np.round(src / 16384.0) * 16384.0).astype(np.float32)
    poster[10:20, 10:30] = 32768.0
    for typ in (1, 2, 3, 4, 5, 6, 7, 8, 9, 10):
        for W, H in ((3, 3), (5, 5), (4, 2), (1, 7), (1, 1)):
            for image in ((src, poster) if typ in (4, 6, 7) else (src,)):
                b = np.empty_like(image)
                assert oracle().orc_statistic(P(image), P(b), 47, 33, ch, typ, W, H) == 0
                expect_ref(b, "ref_statistic", image, OUT, 47, 33, ch, typ, W, H)


@pytest.mark.parametrize("ch", [1, 4])
def test_thumbnail_pixel_path_bit_exact(ch):
    """resize.c:4591 ThumbnailImage: sample (factors > 4) / box (factors > 2) / LanczosSharp cascade."""
    src = make_image(640, 480, ch, seed=9, kind="alpha_blocks" if ch == 4 else "noise")
    for ow, oh in ((64, 48), (100, 75), (200, 150), (320, 240), (400, 300), (640, 480), (31, 23)):
        b = np.empty((oh, ow, ch), np.float32)
        assert oracle().orc_thumbnail(P(src), 640, 480, ch, P(b), ow, oh) == 0
        expect_ref(b, "ref_thumbnail", src, 640, 480, ch, OUT, ow, oh)


@pytest.mark.parametrize("ch", [1, 4])
def test_resize_all_filters_bit_exact(ch):
    src = make_image(47, 33, ch, seed=5, kind="alpha_blocks")
    for filt in [0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16, 17, 18, 19, 20, 21, 22, 23, 24, 25, 26, 27, 28, 29, 30, 31, 32, 33]:
        for ow, oh in ((23, 16), (24, 17), (94, 66), (47, 10), (13, 33)):
            b = np.empty((oh, ow, ch), np.float32)
            assert oracle().orc_resize(P(src), 47, 33, ch, P(b), ow, oh, filt) == 0
            expect_ref(b, "ref_resize", src, 47, 33, ch, OUT, ow, oh, filt)


@pytest.mark.parametrize("name,args", [("Disk:3", ("disk", 3, 1, 0, 0)), ("Octagon:2", ("octagon", 2, 1, 0, 0)),
                                       ("Plus:2", ("plus", 2, 1, 0, 0)), ("Square:1", ("square", 1, 1, 0, 0)),
                                       ("Rectangle:4x2+3+0", ("rectangle", 4, 2, 3, 0))])
def test_morphology_bit_exact(name, args):
    k = util.orc_kernel(*args)
    ref_vals, x, y = util.stored_ref_kernel(name)
    assert (k.x, k.y) == (x, y)
    mine = k.array()
    assert np.array_equal(np.isnan(mine), np.isnan(ref_vals))
    assert np.array_equal(mine[~np.isnan(mine)], ref_vals[~np.isnan(ref_vals)])
    for ch in (1, 2, 4):
        src = make_image(40, 29, ch, seed=3)
        for method, its in ((3, 1), (4, 1), (4, 2), (8, 1), (9, 1), (12, 1), (3, -1),
                            (13, 1), (14, 1), (15, 1), (16, 1), (17, 1), (15, 2), (17, 3)):   # Edge*/TopHat/BottomHat
            expect_ref(util.orc_morphology(src, method, its, [k]), "ref_morphology", src, OUT, 40, 29, ch, method, its,
                       name.encode())


@pytest.mark.parametrize("frm,to", [(23, 11), (23, 26), (23, 21), (11, 23), (26, 23), (21, 23), (26, 11)])
def test_colorspace_bit_exact(frm, to):
    src = make_image(64, 48, 4, seed=8)
    b = src.copy()
    assert oracle().orc_colorspace(P(b), 64, 48, 4, frm, to) == 0
    expect_ref(b, "ref_colorspace", InOut(src), 64, 48, 4, frm, to)


def ref_kernel_list(string):
    """The reference's own (expanded) kernel list for a kernel string, as oracle kernels."""
    out, idx = [], 0
    while True:
        k = util.stored_ref_kernel(string, idx)
        if k is None:
            return out
        out.append(util.orc_kernel_from_array(k[0], k[1], k[2]))
        idx += 1


HMT_CASES = [(18, 1, "Corners"), (18, 1, "LineEnds"), (18, 2, "3x3:1,1,1 0,1,0 -,0,-"), (18, 1, "Peaks:1.9"),
             (18, 3, "Edges"), (19, 1, "Skeleton:2"), (19, -1, "Skeleton"), (19, 2, "LineEnds"), (19, 1, "ThinSE:482"),
             (20, 1, "ConvexHull"), (20, 3, "Corners"), (5, 1, "Disk:2"), (6, 1, "Disk:2"), (5, 2, "Rectangle:3x2+0+1"),
             (6, 3, "Octagon:2"), (10, 1, "Disk:2.5"), (11, 1, "Rectangle:4x3+1+0"), (11, 2, "Diamond:2"),
             (7, 1, "Euclidean:2"), (7, 4, "Chebyshev:1"), (7, -1, "Manhattan")]


@pytest.mark.parametrize("method,its,name", HMT_CASES)
def test_hit_and_miss_intensity_distance_bit_exact(method, its, name):
    """HitAndMiss / Thinning / Thicken (morphology.c:3037-3083, lists united with Lighten or re-iterated, the whole
    method iterated: :3722-3729), Erode / Dilate / Open / CloseIntensity (:3084-3137: a whole pixel is copied),
    IterativeDistance (:3138-3181) -- the kernels are the reference's own expansion of the kernel string."""
    kernels = ref_kernel_list(name)
    assert kernels
    for ch, kind in ((1, "binary"), (3, "binary"), (4, "alpha_blocks"), (2, "noise"), (3, "hdr")):
        if method == 7 and kind == "hdr":
            continue
        src = make_image(53, 37, ch, seed=40 + ch, kind=kind)
        b = util.orc_morphology(src, method, its, kernels)
        expect_ref(b, "ref_morphology", src, OUT, 53, 37, ch, method, its, name.encode())


def hexcone_image(kind):
    """Noise plus the pixels the hexcone formulae branch on: grays, black, white, primaries, two-way ties of the
    maximum / minimum, hues on the sector boundaries."""
    src = make_image(64, 48, 4, seed=8, kind=kind)
    special = np.array([[0, 0, 0], [65535, 65535, 65535], [32768, 32768, 32768], [65535, 0, 0], [0, 65535, 0],
                        [0, 0, 65535], [65535, 65535, 0], [0, 65535, 65535], [65535, 0, 65535], [40000, 40000, 100],
                        [100, 40000, 40000], [40000, 100, 40000], [1, 0, 0], [65535, 65534, 65535], [10922.5, 0, 0],
                        [21845, 30000, 30000], [43690, 65535, 65535], [54612.5, 20000, 50000], [0, 65535, 32767.5],
                        [16383.75, 65535, 65535], [65535, 32768, 16384]], np.float32)
    src[0, :len(special), :3] = special
    return src


HEXCONE = [4, 5, 6, 7, 8, 9, 10]      # HCL, HCLp, HSB, HSI, HSL, HSV, HWB (colorspace.h:27-67)


@pytest.mark.parametrize("cs", HEXCONE)
@pytest.mark.parametrize("kind", ["noise", "hdr"])
def test_hexcone_colorspaces_bit_exact(cs, kind):
    """colorspace.c:958-1054 / :2296-2390 with the gem-style conversions of colorspace-private.h: forward from sRGB,
    inverse from arbitrary component values, and a hop between two hexcone spaces (through sRGB, :1773)."""
    src = hexcone_image(kind)
    for frm, to in ((23, cs), (cs, 23), (cs, 8 if cs != 8 else 9)):
        b = src.copy()
        assert oracle().orc_colorspace(P(b), 64, 48, 4, frm, to) == 0
        expect_ref(b, "ref_colorspace", InOut(src), 64, 48, 4, frm, to, nan_equal=True)


# (filter, "-define" string as the CLI would set it, the same settings as values)
FILTER_DEFINES = [
    (22, "filter:blur=0.8", dict(blur=0.8)),
    (22, "filter:lobes=2", dict(lobes=2)),
    (22, "filter:lobes=5;filter:blur=1.1", dict(lobes=5, blur=1.1)),
    (8, "filter:sigma=0.75", dict(sigma=0.75)),
    (8, "filter:sigma=0.3;filter:support=1.25", dict(sigma=0.3, support=1.25)),
    (16, "filter:kaiser-beta=4.5", dict(kaiser_beta=4.5)),
    (16, "filter:kaiser-alpha=2.0", dict(kaiser_beta=2.0 * 3.14159265358979323846264338327950288419716939937510)),
    (16, "filter:alpha=8;filter:lobes=4", dict(kaiser_beta=8.0, lobes=4)),
    (10, "filter:b=0.5", dict(b=0.5)),
    (10, "filter:c=0.75", dict(c=0.75)),
    (12, "filter:b=0.2;filter:c=0.6", dict(b=0.2, c=0.6)),
    (3, "filter:window=Hann", dict(window=5)),
    (22, "filter:window=Blackman;filter:win-support=2", dict(window=7, win_support=2.0)),
    (11, "filter:filter=true;filter:window=Welch", dict(window=17, keep_filter=1)),
    (13, "filter:lobes=2", dict(lobes=2)),
    (13, "filter:lobes=20;filter:blur=0.9", dict(lobes=20, blur=0.9)),
    (21, "filter:support=3", dict(support=3.0)),
    (14, "filter:support=2.5;filter:win-support=4", dict(support=2.5, win_support=4.0)),
    (22, "filter:filter=Mitchell", dict()),                 # not a truthy string: ignored by this version (resize.c:1000)
]


@pytest.mark.parametrize("case", range(len(FILTER_DEFINES)))
def test_resize_expert_settings_bit_exact(case):
    """AcquireResizeFilter's "filter:*" artifacts (resize.c:999-1226): the reference with the artifacts set as the CLI's
    -define does, the oracle with the same settings as values."""
    filt, defines, values = FILTER_DEFINES[case]
    opts = util.FilterOptions.of(**values)
    for ch in (3, 4):
        src = make_image(47, 33, ch, seed=5 + case, kind="alpha_blocks" if ch == 4 else "noise")
        for ow, oh in ((23, 16), (94, 66), (47, 10), (31, 33)):
            b = np.empty((oh, ow, ch), np.float32)
            assert oracle().orc_resize_ex(P(src), 47, 33, ch, P(b), ow, oh, filt, C.byref(opts)) == 0
            expect_ref(b, "ref_resize_defines", src, 47, 33, ch, OUT, ow, oh, filt, defines.encode())


XYZ_FAMILY = [12, 13, 14, 16, 17, 25, 34, 35, 36, 37, 38, 39, 40]   # (34 = Jzazbz) LCH, LCHab, LCHuv, LMS, Luv, xyY, DisplayP3, Adobe98, ProPhoto, Oklab, Oklch, CAT02LMS


@pytest.mark.parametrize("cs", XYZ_FAMILY)
@pytest.mark.parametrize("kind", ["noise", "hdr"])
def test_xyz_family_colorspaces_bit_exact(cs, kind):
    """The generic branch's XYZ-derived spaces (colorspace-private.h:53-130, :600-760, :938-1272): forward, inverse and a
    hop to another space of the family."""
    src = hexcone_image(kind)
    for frm, to in ((23, cs), (cs, 23), (cs, 17 if cs != 17 else 25)):
        b = src.copy()
        assert oracle().orc_colorspace(P(b), 64, 48, 4, frm, to) == 0
        expect_ref(b, "ref_colorspace", InOut(src), 64, 48, 4, frm, to, nan_equal=True)


# (colourspace, settings as the CLI would give them, the same settings as values)
COLORSPACE_SETTINGS = [
    (11, "color:illuminant=D50", dict(illuminant="D50")),
    (11, "color:illuminant=A", dict(illuminant="A")),
    (13, "color:illuminant=F11", dict(illuminant="F11")),
    (14, "color:illuminant=E", dict(illuminant="E")),
    (12, "color:illuminant=C", dict(illuminant="C")),
    (17, "color:illuminant=D75", dict(illuminant="D75")),
    (17, "color:illuminant=nonsense", dict()),                      # unparsable: UndefinedIlluminant == D65 (color.h:42)
    (34, "white-luminance=203", dict(white_luminance=203.0)),
    (34, "white-luminance=1000", dict(white_luminance=1000.0)),
    (15, "", dict()),
    (15, "gamma=2.2", dict()),          # SetImageProperty diverts "gamma" to image->gamma (property.c:4583): no effect
    (15, "film-gamma=0.5;reference-black=64;reference-white=940", dict(film_gamma=0.5, reference_black=64.0, reference_white=940.0)),
    (15, "film-gamma=0.65;reference-white=700", dict(film_gamma=0.65, reference_white=700.0)),
    (28, "", dict()),
]


@pytest.mark.parametrize("case", range(len(COLORSPACE_SETTINGS)))
@pytest.mark.parametrize("kind", ["noise", "hdr"])
def test_colorspace_settings_bit_exact(case, kind):
    """The settings TransformImageColorspace reads from the image -- "color:illuminant" (colorspace.c:761-773), "white-luminance"
    (:996), "film-gamma" / "reference-black" / "reference-white" (:1085-1095) -- and the two LUT spaces that
    complete the switch: Log (:1055-1163, :2391-2500) and YCC (:1347-1389, :2681-2711; the oracle regenerates the 1389-entry
    PhotoYCC table from its rule, so this also pins that rule)."""
    cs, defines, values = COLORSPACE_SETTINGS[case]
    opts = util.ColorspaceOptions.of(**values)
    src = hexcone_image(kind)
    src[0, :6, :3] = [[0, 0, 0], [65535, 65535, 65535], [0.4, 0.5, 0.6], [65534.6, 70000, -3], [1179.4, 1179.6, 1180.5], [40092, 35209, 100]]
    for frm, to in ((23, cs), (cs, 23), (cs, 26), (21, cs)):
        b = src.copy()
        assert oracle().orc_colorspace_ex(P(b), 64, 48, 4, frm, to, C.byref(opts)) == 0
        expect_ref(b, "ref_colorspace_defines", InOut(src), 64, 48, 4, frm, to, defines.encode(), nan_equal=True)


@pytest.mark.parametrize("kind", ["alpha_blocks", "hdr"])
def test_difference_methods_bit_exact_on_awkward_pixels(kind):
    """EdgeIn/EdgeOut/Edge/TopHat/BottomHat end in CompositeImage(Difference) (morphology.c:3995-4012):
    transparent regions (PerceptibleReciprocal), values outside 0..QuantumRange (ClampPixel)."""
    k = util.orc_kernel("disk", 3, 1, 0, 0)
    for ch in (2, 3, 4):
        src = make_image(61, 43, ch, seed=21, kind=kind)
        for method in (13, 14, 15, 16, 17):
            expect_ref(util.orc_morphology(src, method, 1, [k]), "ref_morphology", src, OUT, 61, 43, ch, method, 1, b"Disk:3")


THRESHOLD_CASES = [(0, 32768.0, ""), (0, 12345.678, ""), (3, 0.0, ""), (1, 0.0, "50%"), (2, 0.0, "50%"),
                   (1, 0.0, "20000,30000,40000"), (2, 0.0, "20%,30%,40%,50%"), (1, 0.0, "30000,20000,40000,35000"),
                   (2, 0.0, "45000")]


@pytest.mark.parametrize("ch", [1, 2, 3, 4])
@pytest.mark.parametrize("kind", ["noise", "hdr", "gradient"])
def test_threshold_point_ops_bit_exact(ch, kind):
    """threshold.c BilevelImage / BlackThresholdImage / WhiteThresholdImage / ClampImage, incl. samples
    exactly on the threshold and the gray -> sRGB promotion the black/white operators apply."""
    src = make_image(97, 61, ch, seed=5, kind=kind)
    src[0, :10, :] = 32768.0
    src[1, :10, :] = 32767.5
    for op, thr, spec in THRESHOLD_CASES:
        if op in (1, 2) and ch < 3:
            # channel count changed: gray image promoted to sRGB (threshold.c:949)
            expect_ref(None, "ref_threshold", InOut(src), 97, 61, ch, op, thr, spec.encode(), rc=-2)
            continue
        got = util.orc_threshold(src, op, [thr] if op in (0, 3) else util.parse_thresholds(spec))
        expect_ref(got, "ref_threshold", InOut(src), 97, 61, ch, op, thr, spec.encode())


MATRIX_SPACES = [1, 18, 19, 20, 27, 29, 30, 31, 32]   # CMY, OHTA, Rec601YCbCr, Rec709YCbCr, YCbCr, YDbDr, YIQ, YPbPr, YUV


@pytest.mark.parametrize("cs", MATRIX_SPACES)
@pytest.mark.parametrize("kind", ["noise", "hdr"])
def test_matrix_and_lut_colorspaces_bit_exact(cs, kind):
    """Generic-branch matrix spaces and the LUT branch (colorspace.c:1229-1494, :2560-2830), both
    directions and chained through sRGB (colorspace.c:1773), incl. out-of-range samples (HDRI) that the
    16-bit map quantisation clamps."""
    for ch in (3, 4):
        src = make_image(64, 48, ch, seed=8, kind=kind)
        src[0, :4, :3] = [[0, 0, 0], [65535, 65535, 65535], [0.4, 0.5, 0.6], [65534.6, 70000, -3]]
        for frm, to in ((23, cs), (cs, 23), (cs, 11), (21, cs), (cs, 18 if cs != 18 else 30)):
            b = src.copy()
            assert oracle().orc_colorspace(P(b), 64, 48, ch, frm, to) == 0
            expect_ref(b, "ref_colorspace", InOut(src), 64, 48, ch, frm, to)


def test_thread_count_independence():
    """SURVEY 8c: results do not depend on the OpenMP thread count -- the reference's run on 1 and on 4 threads, and
    the oracle's on as many, all agree."""
    src = make_image(128, 96, 4, seed=1)
    outs = []
    try:
        for n in (1, 4):
            oracle().orc_set_threads(n)
            b = np.empty_like(src)
            assert oracle().orc_blur(P(src), P(b), 128, 96, 4, 0.0, 2.0) == 0
            expect_ref(b, "ref_blur", src, OUT, 128, 96, 4, 0.0, 2.0, threads=n)
            outs.append(b)
    finally:
        oracle().orc_set_threads(os.cpu_count() or 1)
    assert max_ulp(outs[0], outs[1]) == 0


@pytest.mark.parametrize("ch", [1, 2, 3, 4])
@pytest.mark.parametrize("kind", ["noise", "gradient", "hdr"])
@pytest.mark.parametrize("sync", [1, 0])
def test_equalize_bit_exact(ch, kind, sync):
    """EqualizeImage (enhance.c:2040): histogram / running sums / table lookup restated; integer counts and one division
    per table entry, so the restatement must reproduce the reference bit for bit."""
    src = util.make_image(97, 61, ch, seed=31, kind=kind)
    a = src.copy()
    assert util.oracle().orc_equalize(util.P(a), 97, 61, ch, sync) == 0
    expect_ref(a, "ref_equalize", InOut(src), 97, 61, ch, sync)
    assert not np.array_equal(a, src)


@pytest.mark.parametrize("ch", [1, 3, 4])
@pytest.mark.parametrize("radius,sigma", [(0.0, 1.0), (0.0, 2.0), (2.0, 0.7)])
def test_emboss_bit_exact(ch, radius, sigma):
    """EmbossImage (effect.c:1600): inline anti-diagonal kernel + ConvolveImage + EqualizeImage."""
    src = util.make_image(83, 59, ch, seed=32, kind="alpha_blocks" if ch == 4 else "noise")
    a = np.empty_like(src)
    assert util.oracle().orc_emboss(util.P(src), util.P(a), 83, 59, ch, radius, sigma) == 0
    expect_ref(a, "ref_emboss", src, OUT, 83, 59, ch, radius, sigma)


@pytest.mark.parametrize("ch", [1, 2, 3, 4])
@pytest.mark.parametrize("sizes", [((64, 48), (32, 24)), ((67, 45), (29, 31)), ((40, 30), (100, 75)), ((53, 37), (53, 20)),
                                   ((53, 37), (17, 37)), ((33, 21), (34, 22)), ((100, 3), (7, 9)), ((256, 256), (85, 85))])
def test_scale_image_bit_exact(ch, sizes):
    """ScaleImage (resize.c:4106): the box-scaling state machine restated literally."""
    (w, h), (ow, oh) = sizes
    src = util.make_image(w, h, ch, seed=81, kind="alpha_blocks" if ch in (2, 4) else "noise")
    a = np.empty((oh, ow, ch), np.float32)
    assert util.oracle().orc_scale(util.P(src), w, h, ch, util.P(a), ow, oh) == 0
    expect_ref(a, "ref_scale", src, w, h, ch, OUT, ow, oh)


@pytest.mark.parametrize("ch", [1, 2, 3, 4])
@pytest.mark.parametrize("args", [(0.0, 1.0, 6553.5), (0.0, 2.0, 20000.0), (2.0, 1.0, 1000.0), (0.0, 1.5, 65535.0 * 2)])
def test_selective_blur_bit_exact(ch, args):
    """SelectiveBlurImage (effect.c:3406): contrast-gated Gaussian; gray image clone + double intensities restated."""
    src = util.make_image(61, 43, ch, seed=82, kind="alpha_blocks" if ch in (2, 4) else "gradient")
    a = np.empty_like(src)
    assert util.oracle().orc_selective_blur(util.P(src), util.P(a), 61, 43, ch, *args) == 0
    expect_ref(a, "ref_selective_blur", src, OUT, 61, 43, ch, *args)


@pytest.mark.parametrize("ch", [1, 2, 3, 4])
@pytest.mark.parametrize("fn", ["adaptive_blur", "adaptive_sharpen"])
@pytest.mark.parametrize("args", [(0.0, 1.0), (0.0, 2.0), (3.0, 1.5), (0.0, 0.0)])
def test_adaptive_blur_and_sharpen_bit_exact(ch, fn, args):
    """AdaptiveBlurImage / AdaptiveSharpenImage (effect.c:128 / :447): edge -> auto-level -> blur -> auto-level selects a
    kernel size per pixel."""
    src = util.make_image(75, 52, ch, seed=83, kind="alpha_blocks" if ch in (2, 4) else "gradient")
    a = np.empty_like(src)
    assert getattr(util.oracle(), "orc_" + fn)(util.P(src), util.P(a), 75, 52, ch, *args) == 0
    expect_ref(a, "ref_" + fn, src, OUT, 75, 52, ch, *args)
