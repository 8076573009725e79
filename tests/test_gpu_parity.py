"""Parity of the CUDA path (through the C-ABI) against the oracle on seeded inputs.

Bar (BASELINE.json north_star): bit-exact for erode/dilate (selection ops), <= 1 ULP of
the float Quantum for convolution / resize / colourspace.
"""
import ctypes as C

import numpy as np
import pytest

import util
from util import P, make_image, max_ulp, oracle

pytestmark = pytest.mark.gpu

im = pytest.importorskip("imagemagick_b200")


def _dev(a: np.ndarray):
    import torch
    return im.Image(torch.from_numpy(a).cuda())


def _host(img) -> np.ndarray:
    return img.pixels.cpu().numpy() if img.on_device else img.pixels


def orc(fn, src, *args):
    h, w, ch = src.shape
    dst = np.empty_like(src)
    assert getattr(oracle(), fn)(P(src), P(dst), w, h, ch, *args) == 0
    return dst


SIZES = [(67, 45), (256, 131), (1, 1), (5, 300), (300, 3)]


@pytest.mark.parametrize("ch", [1, 2, 3, 4])
@pytest.mark.parametrize("kind", ["noise", "alpha_blocks", "hdr"])
@pytest.mark.parametrize("radius,sigma", [(0.0, 2.0), (0.0, 4.0), (0.0, 0.5), (3.0, 1.5), (0.0, 1.0), (0.0, 3.0)])
def test_blur_host_path(ch, kind, radius, sigma):
    for (w, h) in SIZES[:3]:
        src = make_image(w, h, ch, seed=w * 7 + ch, kind=kind)
        want = orc("orc_blur", src, radius, sigma)
        got = im.BlurImage(im.Image(src), radius, sigma).pixels
        assert max_ulp(got, want) <= 1, (w, h, ch, kind, radius, sigma)


@pytest.mark.parametrize("ch", [1, 2, 3, 4])
@pytest.mark.parametrize("sigma", [2.0, 4.0, 6.0, 8.0])
def test_blur_device_path(ch, sigma):
    for (w, h) in SIZES:
        src = make_image(w, h, ch, seed=w + h + ch)
        want = orc("orc_blur", src, 0.0, sigma)
        got = _host(im.BlurImage(_dev(src), 0.0, sigma))
        assert max_ulp(got, want) <= 1, (w, h, ch, sigma)


def test_blur_config1_1024_rgba_sigma2():
    """BASELINE.json configs[0]: 1024x1024 RGBA GaussianBlur sigma=2 (BlurImage(0,2))."""
    src = make_image(1024, 1024, 4, seed=42)
    want = orc("orc_blur", src, 0.0, 2.0)
    got = _host(im.BlurImage(_dev(src), 0.0, 2.0))
    d = util.ulp_distance(got, want)
    assert d.max() <= 1
    assert (d == 0).mean() > 0.999


def test_blur_wide_kernel_falls_back_to_generic():
    src = make_image(200, 90, 4, seed=3)
    want = orc("orc_blur", src, 0.0, 12.0)       # 97 taps > templated sizes
    got = _host(im.BlurImage(_dev(src), 0.0, 12.0))
    assert max_ulp(got, want) <= 1


@pytest.mark.parametrize("ch", [1, 3, 4])
@pytest.mark.parametrize("sigma", [1.0, 2.0])
def test_gaussian_blur_2d(ch, sigma):
    src = make_image(97, 61, ch, seed=11, kind="alpha_blocks")
    want = orc("orc_gaussian_blur", src, 0.0, sigma)
    assert max_ulp(im.GaussianBlurImage(im.Image(src), 0.0, sigma).pixels, want) <= 1
    assert max_ulp(_host(im.GaussianBlurImage(_dev(src), 0.0, sigma)), want) <= 1


@pytest.mark.parametrize("kind", ["noise", "alpha_blocks", "hdr"])
@pytest.mark.parametrize("sigma", [0.5, 1.0, 2.0, 3.0, 4.0])
def test_gaussian_blur_2d_rank1_path(kind, sigma, monkeypatch):
    """RGBA rank-1 kernels run as row pass (raw double sums) + column pass; both that path and the
    direct kw*kh kernel must agree with the oracle's 2-D MorphologyPrimitive."""
    for (w, h) in ((97, 61), (300, 5), (3, 200), (1, 1), (640, 130)):
        src = make_image(w, h, 4, seed=w + 3, kind=kind)
        want = orc("orc_gaussian_blur", src, 0.0, sigma)
        n0 = im.launch_count()
        got = _host(im.GaussianBlurImage(_dev(src), 0.0, sigma))
        launches = im.launch_count() - n0
        assert max_ulp(got, want) <= 1, (w, h, kind, sigma)
        util.set_option("no_rank1", 1)
        n0 = im.launch_count()
        direct = _host(im.GaussianBlurImage(_dev(src), 0.0, sigma))
        assert im.launch_count() - n0 == 1
        util.set_option("no_rank1", 0)
        assert max_ulp(direct, want) <= 1
        assert launches == 2          # the separable path was taken


def test_rank1_user_kernel_and_non_rank1_neighbour():
    src = make_image(150, 90, 4, seed=77, kind="alpha_blocks")
    col = np.array([1.0, 3.0, 2.0, 0.5, 0.25])
    row = np.array([0.5, 2.0, 1.0])
    vals = np.outer(col, row)
    for (x, y) in ((1, 2), (0, 4), (2, 0)):
        k = util.orc_kernel_from_array(vals, x, y)
        ks = f"3x5+{x}+{y}: " + " ".join(",".join(repr(float(v)) for v in r) for r in vals)
        want = util.orc_morphology(src, im.ConvolveMorphology, 1, [k])
        n0 = im.launch_count()
        got = _host(im.MorphologyImage(_dev(src), im.ConvolveMorphology, 1, ks))
        assert im.launch_count() - n0 == 2
        assert max_ulp(got, want) <= 1, (x, y)
    vals2 = vals.copy()
    vals2[2, 1] += 1e-9                      # no longer rank 1 -> direct kernel
    k = util.orc_kernel_from_array(vals2, 1, 2)
    ks = "3x5+1+2: " + " ".join(",".join(repr(float(v)) for v in r) for r in vals2)
    n0 = im.launch_count()
    got = _host(im.MorphologyImage(_dev(src), im.ConvolveMorphology, 1, ks))
    assert im.launch_count() - n0 == 1
    assert max_ulp(got, util.orc_morphology(src, im.ConvolveMorphology, 1, [k])) <= 1


@pytest.mark.parametrize("ch", [1, 2, 3, 4])
@pytest.mark.parametrize("kind", ["noise", "alpha_blocks"])
def test_sharpen_and_edge(ch, kind):
    """SharpenImage / EdgeImage: kernels with negative taps through the generic 2-D convolution."""
    src = make_image(131, 77, ch, seed=61 + ch, kind=kind)
    for rad, sig in ((0.0, 1.0), (2.0, 0.7)):
        want = orc("orc_sharpen", src, rad, sig)
        assert max_ulp(_host(im.SharpenImage(_dev(src), rad, sig)), want) <= 1, (rad, sig)
    for rad in (0.0, 1.0):
        want = orc("orc_edge", src, rad)
        assert max_ulp(_host(im.EdgeImage(_dev(src), rad)), want) <= 1, rad
    assert max_ulp(im.SharpenImage(im.Image(src), 0.0, 1.0).pixels, orc("orc_sharpen", src, 0.0, 1.0)) <= 1


@pytest.mark.parametrize("ch", [1, 2, 3, 4])
@pytest.mark.parametrize("kind", ["noise", "alpha_blocks", "hdr"])
def test_motion_blur(ch, kind):
    """MotionBlurImage (effect.c:2347): reference-ordered unfused double accumulation => expected bit exact; bar 1 ULP."""
    src = make_image(131, 77, ch, seed=81 + ch, kind=kind)
    for rad, sig, ang in ((0, 2, 0), (0, 2, 45), (0, 3, 90), (0, 1.5, -30), (0, 4, 180), (5, 2, 270), (0, 2, 123.4)):
        want = orc("orc_motion_blur", src, float(rad), float(sig), float(ang))
        got = _host(im.MotionBlurImage(_dev(src), rad, sig, ang))
        assert max_ulp(got, want) <= 1, (rad, sig, ang, max_ulp(got, want))
    got = im.MotionBlurImage(im.Image(src), 0, 2, 30).pixels
    assert max_ulp(got, orc("orc_motion_blur", src, 0.0, 2.0, 30.0)) <= 1


@pytest.mark.parametrize("ch", [1, 2, 3, 4])
def test_unsharp(ch):
    src = make_image(120, 77, ch, seed=5)
    want = orc("orc_unsharp", src, 0.0, 2.0, 1.5, 0.02)
    got = _host(im.UnsharpMaskImage(_dev(src), 0.0, 2.0, 1.5, 0.02))
    d = util.ulp_distance(got, want)
    assert d.max() <= 1                      # SURVEY 8d: <= 1 ULP ...
    assert (d == 0).mean() > 0.9999
    passthrough = want == src                # ... and the |2d| < QR*threshold branch returns the input itself: 0 ULP
    assert passthrough.mean() > 0.005        # the branch is exercised
    assert np.array_equal(got[passthrough], src[passthrough])
    # the fused epilogue of the column pass and the separate point pass are the same arithmetic on the same
    # float-rounded blur: identical bits
    util.set_option("no_fused_unsharp", 1)
    unfused = _host(im.UnsharpMaskImage(_dev(src), 0.0, 2.0, 1.5, 0.02))
    util.set_option("no_fused_unsharp", 0)
    assert np.array_equal(got, unfused)


KERNELS = [("Disk:3", ("disk", 3, 1, 0, 0)), ("Disk:1.5", ("disk", 1.5, 1, 0, 0)), ("Square:2", ("square", 2, 1, 0, 0)),
           ("Diamond:2", ("diamond", 2, 1, 0, 0)), ("Octagon:3", ("octagon", 3, 1, 0, 0)),
           ("Plus:2", ("plus", 2, 1, 0, 0)), ("Cross:1", ("cross", 1, 1, 0, 0)),
           ("Rectangle:5x3+1+2", ("rectangle", 5, 3, 1, 2))]


@pytest.mark.parametrize("ch", [1, 2, 3, 4])
@pytest.mark.parametrize("name,args", KERNELS)
def test_erode_dilate_bit_exact(ch, name, args):
    src = make_image(83, 59, ch, seed=17, kind="hdr" if ch == 3 else "noise")
    k = util.orc_kernel(*args)
    for method, its in ((im.ErodeMorphology, 1), (im.DilateMorphology, 1), (im.DilateMorphology, 3),
                        (im.OpenMorphology, 1), (im.CloseMorphology, 1), (im.SmoothMorphology, 1)):
        want = util.orc_morphology(src, method, its, [k])
        got = _host(im.MorphologyImage(_dev(src), method, its, name))
        assert max_ulp(got, want) == 0, (name, ch, method, its)
        got_h = im.MorphologyImage(im.Image(src), method, its, name).pixels
        assert max_ulp(got_h, want) == 0


STREAM_SHAPES = [("Disk:1", ("disk", 1, 1, 0, 0)), ("Disk:2", ("disk", 2, 1, 0, 0)), ("Disk:2.5", ("disk", 2.5, 1, 0, 0)),
                 ("Disk:3", ("disk", 3, 1, 0, 0)), ("Disk:3.5", ("disk", 3.5, 1, 0, 0)), ("Disk:4", ("disk", 4, 1, 0, 0)),
                 ("Disk:4.5", ("disk", 4.5, 1, 0, 0)), ("Disk:5", ("disk", 5, 1, 0, 0)), ("Square:1", ("square", 1, 1, 0, 0)),
                 ("Square:3", ("square", 3, 1, 0, 0)), ("Square:4", ("square", 4, 1, 0, 0)),
                 ("Diamond:3", ("diamond", 3, 1, 0, 0)), ("Diamond:4", ("diamond", 4, 1, 0, 0)),
                 ("Diamond:5", ("diamond", 5, 1, 0, 0)), ("Octagon:2", ("octagon", 2, 1, 0, 0)),
                 ("Octagon:4", ("octagon", 4, 1, 0, 0)), ("Octagon:5", ("octagon", 5, 1, 0, 0)),
                 ("Plus:3", ("plus", 3, 1, 0, 0)), ("Plus:4", ("plus", 4, 1, 0, 0))]


@pytest.mark.parametrize("ch", [1, 4])
@pytest.mark.parametrize("name,args", STREAM_SHAPES)
def test_erode_dilate_streaming_kernel(ch, name, args, monkeypatch):
    """Built-in structuring elements take the register-streaming kernel (morph_stream.cu): bit exact against
    the oracle and against the generic kernel, on widths around the 32-2R lane groups and strips taller
    than one CTA strip."""
    k = util.orc_kernel(*args)
    for (w, h) in ((83, 59), (1, 1), (3, 140), (22, 7), (23, 67), (300, 150)):
        src = make_image(w, h, ch, seed=w + h, kind="hdr" if w == 23 else "noise")
        for method in (im.ErodeMorphology, im.DilateMorphology):
            want = util.orc_morphology(src, method, 1, [k])
            got = _host(im.MorphologyImage(_dev(src), method, 1, name))
            assert max_ulp(got, want) == 0, (name, ch, method, w, h)
    src = make_image(131, 97, ch, seed=5)
    got = _host(im.MorphologyImage(_dev(src), im.DilateMorphology, 1, name))
    util.set_option("no_morph_stream", 1)
    generic = _host(im.MorphologyImage(_dev(src), im.DilateMorphology, 1, name))
    assert max_ulp(got, generic) == 0


def test_dilate_until_convergence_and_changed_count():
    src = make_image(64, 48, 1, seed=9, kind="binary")
    k = util.orc_kernel("diamond", 1, 1, 0, 0)
    want = util.orc_morphology(src, im.DilateMorphology, -1, [k])
    got = _host(im.MorphologyImage(_dev(src), im.DilateMorphology, -1, "Diamond:1"))
    assert max_ulp(got, want) == 0
    dst = np.empty_like(src)
    changed_ref = oracle().orc_morphology_primitive(P(src), P(dst), 64, 48, 1, im.ErodeMorphology, C.byref(k), 0.0)
    out, changed = im.MorphologyPrimitive(_dev(src), im.ErodeMorphology, "Diamond:1")
    assert changed == changed_ref
    assert max_ulp(_host(out), dst) == 0


@pytest.mark.parametrize("ch", [1, 4])
def test_user_kernel_convolve_and_correlate(ch):
    src = make_image(90, 70, ch, seed=23)
    vals = np.array([[1.0, 2.0, 0.5], [0.0, -1.0, np.nan], [3.0, 0.25, -2.0]])
    k = util.orc_kernel_from_array(vals, 0, 2)
    ks = "3x3+0+2: 1,2,0.5 0,-1,nan 3,0.25,-2"
    for method in (im.ConvolveMorphology, im.CorrelateMorphology):
        want = util.orc_morphology(src, method, 1, [k])
        got = _host(im.MorphologyImage(_dev(src), method, 1, ks))
        assert max_ulp(got, want) <= 1, (ch, method)
    want = util.orc_morphology(src, im.ConvolveMorphology, 1, [k], bias=100.0)
    got = _host(im.MorphologyImage(_dev(src), im.ConvolveMorphology, 1, ks, bias=100.0))
    assert max_ulp(got, want) <= 1


@pytest.mark.parametrize("ch", [1, 2, 3, 4])
def test_sample_image_bit_exact(ch):
    src = make_image(131, 77, ch, seed=9)
    for ow, oh in ((65, 38), (66, 39), (262, 154), (131, 40), (50, 77), (300, 20), (1, 1), (131, 77), (7, 5), (1000, 3)):
        want = np.empty((oh, ow, ch), np.float32)
        assert oracle().orc_sample(P(src), 131, 77, ch, P(want), ow, oh) == 0
        got = _host(im.SampleImage(_dev(src), ow, oh))
        assert np.array_equal(got.view(np.int32), want.view(np.int32)), (ow, oh)
    got = im.SampleImage(im.Image(src), 40, 30).pixels
    want = np.empty((30, 40, ch), np.float32)
    assert oracle().orc_sample(P(src), 131, 77, ch, P(want), 40, 30) == 0
    assert np.array_equal(got.view(np.int32), want.view(np.int32))
    # the offsets are exact at awkward ratios and large sizes: (j + 0.5 - eps) * in / out evaluated in IEEE double
    big = make_image(4099, 3, ch, seed=2)
    want = np.empty((2, 3001, ch), np.float32)
    assert oracle().orc_sample(P(big), 4099, 3, ch, P(want), 3001, 2) == 0
    assert np.array_equal(_host(im.SampleImage(_dev(big), 3001, 2)).view(np.int32), want.view(np.int32))


@pytest.mark.parametrize("ch", [1, 4])
def test_thumbnail_pixel_path(ch):
    """ThumbnailImage's cascade: the sample stage is exact; each of the (up to two) resize stages is a <= 1 ULP
    operator fed by the previous stage, so the cascade is pinned stage by stage on the product's own intermediates
    and end to end with the corresponding budget."""
    src = make_image(640, 480, ch, seed=9, kind="alpha_blocks" if ch == 4 else "noise")
    for ow, oh in ((64, 48), (100, 75), (200, 150), (320, 240), (400, 300), (640, 480), (31, 23)):
        got = _host(im.ThumbnailImage(_dev(src), ow, oh))
        want = np.empty((oh, ow, ch), np.float32)
        assert oracle().orc_thumbnail(P(src), 640, 480, ch, P(want), ow, oh) == 0
        stages = 1 + (640 // ow > 2 and 480 // oh > 2)
        err = np.abs(got.astype(np.float64) - want.astype(np.float64)).max()
        assert err <= stages * 1.5 * 0.00390625, (ow, oh, err)          # float ULPs at the top of the Quantum range
        # stage-wise: reproduce the cascade from the product's own intermediates, each stage within 1 ULP
        cur = _dev(src)
        if 640 // ow > 4 and 480 // oh > 4:
            cur = im.SampleImage(cur, 4 * ow, 4 * oh)
        if 640 // ow > 2 and 480 // oh > 2:
            cur = im.ResizeImage(cur, 2 * ow, 2 * oh, im.BoxFilter)
        if (ow, oh) != (640, 480):
            mid = np.ascontiguousarray(_host(cur))
            last = np.empty((oh, ow, ch), np.float32)
            assert oracle().orc_resize(P(mid), mid.shape[1], mid.shape[0], ch, P(last), ow, oh, 23) == 0
            assert max_ulp(got, last) <= 1, (ow, oh)
    assert max_ulp(im.ThumbnailImage(im.Image(src), 100, 75).pixels, _host(im.ThumbnailImage(_dev(src), 100, 75))) == 0


FILTERS = [1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16, 17, 18, 19, 20, 21, 22, 23, 24, 25, 26, 27, 28, 29, 30, 31, 32, 33]


@pytest.mark.parametrize("ch", [1, 2, 3, 4])
@pytest.mark.parametrize("filt", [22, 12, 0, 3, 11])
def test_resize_shapes(ch, filt):
    src = make_image(131, 77, ch, seed=31, kind="alpha_blocks")
    for (ow, oh) in ((65, 38), (66, 39), (262, 154), (131, 40), (50, 77), (300, 20), (1, 1), (131, 77)):
        want = np.empty((oh, ow, ch), np.float32)
        assert oracle().orc_resize(P(src), 131, 77, ch, P(want), ow, oh, filt) == 0
        got = _host(im.ResizeImage(_dev(src), ow, oh, filt))
        assert max_ulp(got, want) <= 1, (ch, filt, ow, oh)


@pytest.mark.parametrize("filt", FILTERS)
def test_resize_all_filters(filt):
    src = make_image(96, 64, 4, seed=37)
    for (ow, oh) in ((48, 32), (144, 100)):
        want = np.empty((oh, ow, 4), np.float32)
        assert oracle().orc_resize(P(src), 96, 64, 4, P(want), ow, oh, filt) == 0
        got = im.ResizeImage(im.Image(src), ow, oh, filt).pixels
        assert max_ulp(got, want) <= 1, (filt, ow, oh)


def _kernel_list(arrays):
    """The same kernel list for both sides: a 'WxH:...;WxH:...' string for the product's parser, oracle kernels (origin
    at the centre) for the checker."""
    parts, orc_list = [], []
    for a in arrays:
        a = np.asarray(a, np.float64)
        h, w = a.shape
        rows = [",".join("nan" if np.isnan(v) else repr(float(v)) for v in row) for row in a]
        parts.append(f"{w}x{h}:" + " ".join(rows))
        orc_list.append(util.orc_kernel_from_array(a, (w - 1) // 2, (h - 1) // 2))
    return ";".join(parts), orc_list


_N = np.nan
_CORNER = np.array([[0, 0, _N], [0, 1, 1], [_N, 1, _N]])
_LINE_END = np.array([[0, 0, _N], [0, 1, 1], [0, 0, _N]])
_THIN1 = np.array([[0, 0, 0], [_N, 1, _N], [1, 1, 1]])
_THIN2 = np.array([[_N, 0, 0], [1, 1, 0], [_N, 1, _N]])
_DISK2 = np.array([[_N, 1, 1, 1, _N], [1, 1, 1, 1, 1], [1, 1, 1, 1, 1], [1, 1, 1, 1, 1], [_N, 1, 1, 1, _N]])
_RECT = np.ones((2, 3))
_EUCLID = np.array([[np.hypot(u, v) * 655.35 for u in (-2, -1, 0, 1, 2)] for v in (-2, -1, 0, 1, 2)])
_rot4 = lambda a: [np.rot90(a, k) for k in range(4)]
MORPH_SELECT = [(18, 1, _rot4(_CORNER)), (18, 2, [_LINE_END]), (18, 3, _rot4(_LINE_END)),
                (19, 1, _rot4(_THIN1) + _rot4(_THIN2)), (19, -1, _rot4(_THIN1) + _rot4(_THIN2)), (19, 2, [_THIN1]),
                (20, 1, _rot4(_CORNER)), (20, 3, [_CORNER, _LINE_END]),
                (5, 1, [_DISK2]), (6, 1, [_DISK2]), (5, 2, [_RECT]), (6, 3, [_RECT, _DISK2]), (10, 1, [_DISK2]),
                (11, 1, [_RECT]), (11, 2, [_DISK2]), (7, 1, [_EUCLID]), (7, 4, [_EUCLID]), (7, -1, [_EUCLID])]


@pytest.mark.parametrize("case", range(len(MORPH_SELECT)))
def test_hit_and_miss_intensity_and_distance_bit_exact(case):
    """HitAndMiss / Thinning / Thicken (kernel lists united with Lighten or re-iterated, the whole method iterated until
    nothing changes), Erode / Dilate / Open / CloseIntensity (a whole pixel is selected by its Rec709 intensity),
    IterativeDistance: selections and single double operations => bit exact (morphology.c:3037-3181, :3722-3729, :4016-4052)."""
    method, its, arrays = MORPH_SELECT[case]
    string, kernels = _kernel_list(arrays)
    for ch, kind in ((1, "binary"), (3, "binary"), (4, "alpha_blocks"), (2, "noise"), (3, "hdr"), (4, "noise")):
        if method == 7 and kind == "hdr":
            continue
        src = make_image(83, 59, ch, seed=60 + ch + case, kind=kind)
        want = util.orc_morphology(src, method, its, kernels)
        got = _host(im.MorphologyImage(_dev(src), method, its, string))
        assert max_ulp(got, want) == 0, (method, its, ch, kind)
    src = make_image(40, 31, 4, seed=9, kind="binary")                      # host-buffer entry point
    want = util.orc_morphology(src, method, its, kernels)
    assert max_ulp(im.MorphologyImage(im.Image(src), method, its, string).pixels, want) == 0


HEXCONE = [4, 5, 6, 7, 8, 9, 10]      # HCL, HCLp, HSB, HSI, HSL, HSV, HWB


def _hexcone_image(w, h, ch, kind, seed):
    src = make_image(w, h, ch, seed=seed, kind=kind)
    special = np.array([[0, 0, 0], [65535, 65535, 65535], [32768, 32768, 32768], [65535, 0, 0], [0, 65535, 0],
                        [0, 0, 65535], [65535, 65535, 0], [0, 65535, 65535], [65535, 0, 65535], [40000, 40000, 100],
                        [100, 40000, 40000], [40000, 100, 40000], [1, 0, 0], [65535, 65534, 65535], [10922.5, 0, 0],
                        [21845, 30000, 30000], [43690, 65535, 65535], [54612.5, 20000, 50000], [0, 65535, 32767.5],
                        [16383.75, 65535, 65535], [65535, 32768, 16384]], np.float32)
    src[0, :len(special), :3] = special
    return src


@pytest.mark.parametrize("cs", HEXCONE)
@pytest.mark.parametrize("kind", ["noise", "hdr"])
def test_hexcone_colorspaces(cs, kind):
    """HCL / HCLp / HSB / HSL / HSV / HWB are piecewise (sector of the hue, gray and black branches): every operation is
    the reference's unfused double operation => bit exact in both directions, including a hop between two of them.
    HSI takes atan2 / cos from the CUDA math library: <= 1 ULP."""
    bar = 1 if cs == 7 else 0
    for ch in (3, 4):
        src = _hexcone_image(131, 67, ch, kind, seed=90 + cs)
        for frm, to in ((23, cs), (cs, 23), (cs, 8 if cs != 8 else 9)):
            want = src.copy()
            assert oracle().orc_colorspace(P(want), 131, 67, ch, frm, to) == 0
            img = _dev(src.copy())
            img.colorspace = frm
            assert im.TransformImageColorspace(img, to) is True and img.colorspace == to
            got = _host(img)
            assert np.array_equal(np.isnan(got), np.isnan(want)), (ch, frm, to)
            ok = ~np.isnan(want)
            assert max_ulp(np.where(ok, got, np.float32(0)), np.where(ok, want, np.float32(0))) <= bar, (ch, frm, to)
            if ch == 4:
                assert np.array_equal(got[..., 3], src[..., 3])                 # alpha is not part of the transform
    h = im.Image(_hexcone_image(33, 21, 4, kind, seed=3))                       # host-buffer entry point
    want = h.pixels.copy()
    assert oracle().orc_colorspace(P(want), 33, 21, 4, 23, cs) == 0
    im.TransformImageColorspace(h, cs)
    assert max_ulp(h.pixels, want) <= bar


XYZ_FAMILY = [12, 13, 14, 16, 17, 25, 34, 35, 36, 37, 38, 39, 40]   # (34 = Jzazbz) LCH, LCHab, LCHuv, LMS, Luv, xyY, DisplayP3, Adobe98, ProPhoto, Oklab, Oklch, CAT02LMS
POLAR = (12, 13, 14)                            # hue = atan2 of two differences that cancel for achromatic pixels


def _mask_achromatic_hue(got, want, to):
    """LCHab / LCHuv: where the chroma is rounding noise (|C - 0.5| < 1e-9 of the range) the reference's hue is the atan2 of
    two residues of the XYZ chain -- arbitrary, and only a bit-identical chain (glibc pow included) reproduces it."""
    if to not in POLAR:
        return got, want
    got, want = got.copy(), want.copy()
    achromatic = np.abs(want[..., 1].astype(np.float64) - 32767.5) < 1.0e-4
    got[..., 2] = np.where(achromatic, np.float32(0), got[..., 2])
    want[..., 2] = np.where(achromatic, np.float32(0), want[..., 2])
    return got, want



@pytest.mark.parametrize("cs", XYZ_FAMILY)
@pytest.mark.parametrize("kind", ["noise", "hdr"])
def test_xyz_family_colorspaces(cs, kind):
    """Matrix / transfer-curve / chromaticity spaces derived from XYZ (colorspace-private.h:53-130, :600-760, :938-1272):
    smooth functions of the sample, <= 1 ULP like the Lab / XYZ legs they are built from."""
    for ch in (3, 4):
        src = _hexcone_image(131, 67, ch, kind, seed=120 + cs)
        for frm, to in ((23, cs), (cs, 23), (cs, 17 if cs != 17 else 25), (11, cs if cs not in POLAR else 17)):
            want = src.copy()
            assert oracle().orc_colorspace(P(want), 131, 67, ch, frm, to) == 0
            img = _dev(src.copy())
            img.colorspace = frm
            assert im.TransformImageColorspace(img, to) is True and img.colorspace == to
            got, want = _mask_achromatic_hue(_host(img), want, to)
            ok = np.isfinite(want)
            assert np.array_equal(np.isfinite(got), ok), (ch, frm, to)
            d = util.ulp_or_noise(np.where(ok, got, np.float32(0)), np.where(ok, want, np.float32(0)))
            # a hop through two <= 1 ULP legs can add up; single legs must stay within 1 ULP
            assert d.max() <= (1 if 23 in (frm, to) else 4), (ch, frm, to, int(d.max()))
            assert (d == 0).mean() > 0.99, (ch, frm, to, float((d == 0).mean()))


# (colourspace, the image's settings as strings -- what the python mirror / the shim parse --, the same as values)
COLORSPACE_SETTINGS = [
    (11, {"color:illuminant": "D50"}, dict(illuminant="D50")),
    (11, {"color:illuminant": "A"}, dict(illuminant="A")),
    (13, {"color:illuminant": "F11"}, dict(illuminant="F11")),
    (14, {"color:illuminant": "E"}, dict(illuminant="E")),
    (12, {"color:illuminant": "C"}, dict(illuminant="C")),
    (17, {"color:illuminant": "D75"}, dict(illuminant="D75")),
    (17, {"color:illuminant": "nonsense"}, dict()),
    (34, {"white-luminance": "203"}, dict(white_luminance=203.0)),
    (15, {}, dict()),
    (15, {"film-gamma": "0.5", "reference-black": "64", "reference-white": "940"}, dict(film_gamma=0.5, reference_black=64.0, reference_white=940.0)),
    (15, {"film-gamma": "0.65", "reference-white": "700"}, dict(film_gamma=0.65, reference_white=700.0)),
    (28, {}, dict()),
]


@pytest.mark.parametrize("case", range(len(COLORSPACE_SETTINGS)))
@pytest.mark.parametrize("kind", ["noise", "hdr"])
def test_colorspace_settings(case, kind):
    """The settings TransformImageColorspace reads from the image (colorspace.c:761-773 illuminant, :996 white luminance,
    :1085-1095 the Log film settings) and the two table spaces Log (:1055-1163, :2391-2500) and YCC (:1347-1389,
    :2681-2711).  YCC is unfused arithmetic on map indices and a table => bit exact both ways; the forward Log leg is a
    gather indexed by the linearised sample => bit exact; its inverse ends in EncodePixelGamma => <= 1 ULP; the
    illuminant / white-luminance legs are the <= 1 ULP xyz_family kernels with other constants."""
    cs, settings, values = COLORSPACE_SETTINGS[case]
    opts = util.ColorspaceOptions.of(**values)
    for ch in (3, 4):
        src = _hexcone_image(131, 67, ch, kind, seed=160 + case)
        src[1, :6, :3] = [[0, 0, 0], [65535, 65535, 65535], [0.4, 0.5, 0.6], [65534.6, 70000, -3], [1179.4, 1179.6, 1180.5], [40092, 35209, 100]]
        for frm, to in ((23, cs), (cs, 23)):
            want = src.copy()
            assert oracle().orc_colorspace_ex(P(want), 131, 67, ch, frm, to, C.byref(opts)) == 0
            img = _dev(src.copy())
            img.colorspace = frm
            assert im.TransformImageColorspace(img, to, settings=settings) is True and img.colorspace == to
            got, want = _mask_achromatic_hue(_host(img), want, to)
            ok = np.isfinite(want)
            assert np.array_equal(np.isfinite(got), ok), (ch, frm, to)
            got, want = np.where(ok, got, np.float32(0)), np.where(ok, want, np.float32(0))
            exact = cs == 28 or (cs == 15 and to == 15)
            d = util.ulp_distance(got, want) if exact else util.ulp_or_noise(got, want)
            assert d.max() <= (0 if exact else 1), (ch, frm, to, int(d.max()))
            assert (d == 0).mean() > 0.99, (ch, frm, to, float((d == 0).mean()))
        if cs in (15, 28):
            # linear RGB -> cs: the first leg (linear -> sRGB) is a <= 1 ULP operator in front of a quantiser, so pin the
            # second leg on the product's own first leg (as test_matrix_and_lut_colorspaces does)
            mid = _dev(src.copy())
            mid.colorspace = 21
            im.TransformImageColorspace(mid, 23)
            want = _host(mid).copy()
            assert oracle().orc_colorspace_ex(P(want), 131, 67, ch, 23, cs, C.byref(opts)) == 0
            img = _dev(src.copy())
            img.colorspace = 21
            im.TransformImageColorspace(img, cs, settings=settings)
            assert max_ulp(_host(img), want) == 0, (ch, 21, cs)
    h = im.Image(make_image(33, 21, 4, seed=3))                      # host-buffer entry point
    want = h.pixels.copy()
    assert oracle().orc_colorspace_ex(P(want), 33, 21, 4, 23, cs, C.byref(opts)) == 0
    im.TransformImageColorspace(h, cs, settings=settings)
    assert util.ulp_or_noise(h.pixels, want).max() <= (0 if cs in (15, 28) else 1)


EXPERT_RESIZE = [(22, {"filter:blur": "0.8"}, dict(blur=0.8)), (22, {"filter:lobes": "2"}, dict(lobes=2)),
                 (8, {"filter:sigma": "0.75"}, dict(sigma=0.75)), (16, {"filter:kaiser-beta": "4.5"}, dict(kaiser_beta=4.5)),
                 (10, {"filter:b": "0.5"}, dict(b=0.5)), (12, {"filter:b": "0.2", "filter:c": "0.6"}, dict(b=0.2, c=0.6)),
                 (3, {"filter:window": "Hann"}, dict(window=5)),
                 (11, {"filter:filter": "true", "filter:window": "Welch"}, dict(window=17, keep_filter=1)),
                 (13, {"filter:lobes": "5", "filter:blur": "0.9"}, dict(lobes=5, blur=0.9)),
                 (14, {"filter:support": "2.5", "filter:win-support": "4"}, dict(support=2.5, win_support=4.0)),
                 (22, {"filter:lobes": "2", "filter:blur": "1.0"}, dict(lobes=2, blur=1.0))]


@pytest.mark.parametrize("case", range(len(EXPERT_RESIZE)))
def test_resize_with_expert_filter_settings(case):
    """-define filter:* (AcquireResizeFilter, resize.c:999-1226): the python mirror parses the strings like the shim, the
    library builds the reference's weights from the values; integer reductions take the streaming / TMA kernels."""
    import ctypes as C
    filt, artifacts, values = EXPERT_RESIZE[case]
    opts = util.FilterOptions.of(**values)
    for ch in (3, 4):
        src = make_image(256, 192, ch, seed=80 + case, kind="alpha_blocks" if ch == 4 else "noise")
        for (ow, oh) in ((128, 96), (100, 77), (384, 300)):
            want = np.empty((oh, ow, ch), np.float32)
            assert oracle().orc_resize_ex(P(src), 256, 192, ch, P(want), ow, oh, filt, C.byref(opts)) == 0
            got = _host(im.ResizeImage(_dev(src), ow, oh, filt, artifacts=artifacts))
            assert max_ulp(got, want) <= 1, (filt, artifacts, ch, ow, oh)
    src = make_image(64, 48, 4, seed=2)
    want = np.empty((24, 32, 4), np.float32)
    assert oracle().orc_resize_ex(P(src), 64, 48, 4, P(want), 32, 24, filt, C.byref(opts)) == 0
    assert max_ulp(im.ResizeImage(im.Image(src), 32, 24, filt, artifacts=artifacts).pixels, want) <= 1
    # the table cache keys on the settings: the plain filter right after must not see them
    plain = np.empty((24, 32, 4), np.float32)
    assert oracle().orc_resize(P(src), 64, 48, 4, P(plain), 32, 24, filt) == 0
    assert max_ulp(im.ResizeImage(im.Image(src), 32, 24, filt).pixels, plain) <= 1


def test_resize_lanczos_2x_down_2048():
    """configs[2] at 1/8 scale: Lanczos 2x downscale, 1-ULP check against the CPU result."""
    src = make_image(2048, 2048, 4, seed=42)
    want = np.empty((1024, 1024, 4), np.float32)
    assert oracle().orc_resize(P(src), 2048, 2048, 4, P(want), 1024, 1024, 22) == 0
    got = _host(im.ResizeImage(_dev(src), 1024, 1024, im.LanczosFilter))
    d = util.ulp_distance(got, want)
    assert d.max() <= 1
    assert (d == 0).mean() > 0.999


# streaming kernels of resize_stream.cu: integer-ratio reductions (S, N) = (2,12) Lanczos, (2,8) Lanczos2 /
# Mitchell / Catrom, (2,4) Triangle, (3,19), (4,24), (4,16); ragged sizes (rows not a multiple of 32,
# columns not a multiple of 8), several strips per axis, borders through the gather kernels.
@pytest.mark.parametrize("kind", ["noise", "alpha_blocks", "hdr"])
@pytest.mark.parametrize("filt,ratio", [(22, 2), (24, 2), (12, 2), (11, 2), (3, 2), (22, 3), (22, 4), (24, 4), (12, 4)])
def test_resize_streaming_kernels(filt, ratio, kind, monkeypatch):
    ow, oh = 173, 131
    w, h = ow * ratio, oh * ratio
    src = make_image(w, h, 4, seed=97 + filt + ratio, kind=kind)
    want = np.empty((oh, ow, 4), np.float32)
    assert oracle().orc_resize(P(src), w, h, 4, P(want), ow, oh, filt) == 0
    d = _dev(src)
    n0 = im.launch_count()
    got = _host(im.ResizeImage(d, ow, oh, filt))
    streamed = im.launch_count() - n0
    assert max_ulp(got, want) <= 1, (filt, ratio, kind)
    util.set_option("no_resize_stream", 1)
    ref = _host(im.ResizeImage(d, ow, oh, filt))
    assert streamed == 2                          # one launch per axis (borders ride along as extra CTAs)
    assert max_ulp(got, ref) <= 1
    # only one axis reduced: the other axis is a 1:1 pass through the gather kernel
    util.set_option("no_resize_stream", 0)
    want = np.empty((h, ow, 4), np.float32)
    assert oracle().orc_resize(P(src), w, h, 4, P(want), ow, h, filt) == 0
    assert max_ulp(_host(im.ResizeImage(d, ow, h, filt)), want) <= 1


@pytest.mark.parametrize("ch", [3, 4])
@pytest.mark.parametrize("frm,to", [(23, 11), (23, 26), (23, 21), (11, 23), (26, 23), (21, 23), (11, 26)])
def test_colorspace(ch, frm, to):
    src = make_image(128, 96, ch, seed=41)
    src[0, :8, :3] = [0, 1, 2]                        # toe segment of the sRGB curve
    src[1, :8, :3] = [65535, 2650, 2651]
    # values every real image is full of: black, white, mid gray, saturated primaries (cancellation in L = 116 f(Y) - 16)
    src[2, :7, :3] = [[0, 0, 0], [65535, 65535, 65535], [32768, 32768, 32768], [65535, 0, 0], [0, 65535, 0], [0, 0, 65535],
                      [257, 257, 257]]
    if frm == 11:
        src[3, :3, :3] = [[0, 32767.5, 32767.5], [65535, 32767.5, 32767.5], [0, 0, 0]]   # Lab black / white / corner
    want = src.copy()
    assert oracle().orc_colorspace(P(want), 128, 96, ch, frm, to) == 0
    a = im.Image(src.copy(), colorspace=frm)
    assert im.TransformImageColorspace(a, to) is True and a.colorspace == to
    assert max_ulp(a.pixels, want) <= 1, (ch, frm, to)
    b = _dev(src.copy()); b.colorspace = frm
    im.TransformImageColorspace(b, to)
    assert max_ulp(_host(b), want) <= 1
    if ch == 4:
        assert np.array_equal(a.pixels[..., 3], src[..., 3])   # alpha untouched


@pytest.mark.parametrize("cs", [1, 18, 19, 20, 27, 29, 30, 31, 32])
@pytest.mark.parametrize("kind", ["noise", "hdr"])
def test_matrix_and_lut_colorspaces(cs, kind):
    """CMY / YCbCr / YDbDr / YIQ / YPbPr / YUV (generic branch) and OHTA / Rec601YCbCr / Rec709YCbCr (LUT branch):
    unfused double arithmetic in the reference's order => bit exact on the matrix leg; <= 1 ULP when the chain
    passes through Lab / linear RGB."""
    for ch in (3, 4):
        src = make_image(131, 67, ch, seed=70 + cs, kind=kind)
        src[0, :4, :3] = [[0, 0, 0], [65535, 65535, 65535], [0.4, 0.5, 0.6], [65534.6, 70000, -3]]
        for frm, to, bar in ((23, cs, 0), (cs, 23, 0), (cs, 11, 1), (cs, 18 if cs != 18 else 30, 0)):
            want = src.copy()
            assert oracle().orc_colorspace(P(want), 131, 67, ch, frm, to) == 0
            img = _dev(src.copy())
            img.colorspace = frm
            assert im.TransformImageColorspace(img, to) is True and img.colorspace == to
            assert max_ulp(_host(img), want) <= bar, (ch, frm, to)
        # linear RGB -> cs: the first leg (linear -> sRGB) is a <= 1 ULP operator and the matrix leg amplifies a
        # 1-ULP input difference (CMY = QR - r), so pin the exact second leg on the product's own first leg.
        mid = _dev(src.copy())
        mid.colorspace = 21
        im.TransformImageColorspace(mid, 23)
        want = _host(mid).copy()
        assert oracle().orc_colorspace(P(want), 131, 67, ch, 23, cs) == 0
        img = _dev(src.copy())
        img.colorspace = 21
        im.TransformImageColorspace(img, cs)
        assert max_ulp(_host(img), want) == 0, (ch, 21, cs)
    h = im.Image(make_image(33, 21, 4, seed=3))                      # host-buffer entry point
    want = h.pixels.copy()
    assert oracle().orc_colorspace(P(want), 33, 21, 4, 23, cs) == 0
    im.TransformImageColorspace(h, cs)
    assert max_ulp(h.pixels, want) == 0


def test_config4_lab_then_dilate_512():
    """configs[3] at reduced size: sRGB->Lab then 7x7 Disk dilate."""
    src = make_image(512, 512, 4, seed=42)
    want = src.copy()
    assert oracle().orc_colorspace(P(want), 512, 512, 4, 23, 11) == 0
    k = util.orc_kernel("disk", 3, 1, 0, 0)
    want2 = util.orc_morphology(want, im.DilateMorphology, 1, [k])
    a = _dev(src)
    im.TransformImageColorspace(a, im.LabColorspace)
    lab = _host(a)
    assert max_ulp(lab, want) <= 1
    got2 = _host(im.MorphologyImage(_dev(want), im.DilateMorphology, 1, "Disk:3"))
    assert max_ulp(got2, want2) == 0


@pytest.mark.parametrize("ch", [1, 2, 3, 4])
@pytest.mark.parametrize("kind", ["noise", "alpha_blocks", "hdr"])
def test_difference_morphology_methods_bit_exact(ch, kind):
    """EdgeIn / EdgeOut / Edge / TopHat / BottomHat: erode/dilate stages + the Difference composite of
    morphology.c:3995-4012, bit exact (selection ops + unfused double point arithmetic)."""
    src = make_image(150, 97, ch, seed=50 + ch, kind=kind)
    for kname, kargs in (("Disk:3", ("disk", 3, 1, 0, 0)), ("Rectangle:4x2+3+0", ("rectangle", 4, 2, 3, 0))):
        k = util.orc_kernel(*kargs)
        for method, its in ((13, 1), (14, 1), (15, 1), (16, 1), (17, 1), (15, 2), (17, 2)):
            want = util.orc_morphology(src, method, its, [k])
            got = _host(im.MorphologyImage(_dev(src), method, its, kname))
            assert max_ulp(got, want) == 0, (kname, method, its)
    got = im.MorphologyImage(im.Image(src), im.EdgeMorphology, 1, "Disk:3").pixels     # host-buffer entry point
    assert max_ulp(got, util.orc_morphology(src, 15, 1, [util.orc_kernel("disk", 3, 1, 0, 0)])) == 0
    with pytest.raises(im.MagickB200Error) as e:                                        # multi-kernel list: decline
        im.MorphologyImage(_dev(src), im.EdgeMorphology, 1, "Disk:3;Disk:2")
    assert e.value.code == -5


THRESHOLD_CASES = [(0, 32768.0, ""), (0, 12345.678, ""), (3, 0.0, ""), (1, 0.0, "50%"), (2, 0.0, "50%"),
                   (1, 0.0, "20000,30000,40000"), (2, 0.0, "20%,30%,40%,50%"), (1, 0.0, "30000, 20000 ,40000,35000"),
                   (2, 0.0, "45000")]


@pytest.mark.parametrize("ch", [1, 2, 3, 4])
@pytest.mark.parametrize("kind", ["noise", "hdr", "gradient"])
def test_threshold_point_ops_bit_exact(ch, kind):
    """threshold.c point operators: bit exact (north_star: integer morphology / threshold), device and
    host-buffer entry points, samples exactly on the threshold, NaN through ClampImage."""
    src = make_image(203, 77, ch, seed=15 + ch, kind=kind)
    src[0, :10, :] = 32768.0
    src[1, :10, :] = 32767.5
    src[2, 3, 0] = np.nan
    for op, thr, spec in THRESHOLD_CASES:
        def run(img):
            if op == 0:
                return im.BilevelImage(img, thr)
            if op == 3:
                return im.ClampImage(img)
            return (im.BlackThresholdImage if op == 1 else im.WhiteThresholdImage)(img, spec)
        if op in (1, 2) and ch < 3:
            with pytest.raises(im.MagickB200Error) as e:
                run(_dev(src.copy()))
            assert e.value.code == -5                 # decline: the shim leaves it to the CPU path
            continue
        want = util.orc_threshold(src, op, [thr] if op in (0, 3) else util.parse_thresholds(spec.replace(" ", "")))
        d = _dev(src.copy())
        assert run(d) is True
        got = _host(d)
        assert np.array_equal(got.view(np.int32), want.view(np.int32)), (op, thr, spec)
        h = im.Image(src.copy())
        assert run(h) is True
        assert np.array_equal(h.pixels.view(np.int32), want.view(np.int32)), (op, thr, spec)


def test_threshold_declines():
    img = _dev(make_image(16, 16, 4, seed=1))
    img.colorspace = im.RGBColorspace
    for bad in ("50%x20", "a,b", "1,2,3,4,5", ""):
        with pytest.raises(im.MagickB200Error) as e:
            im.BlackThresholdImage(_dev(make_image(16, 16, 4, seed=1)), bad)
        assert e.value.code == -5
    with pytest.raises(im.MagickB200Error) as e:
        im.WhiteThresholdImage(img, "50%")            # linear RGB needs EncodePixelGamma for the intensity
    assert e.value.code == -5


def test_errors_are_loud():
    src = make_image(16, 16, 4)
    with pytest.raises(im.MagickB200Error):
        im.MorphologyImage(_dev(src), 21, 1, "Disk:1")                    # Distance: sequential two-pass primitive -> decline
    with pytest.raises(im.MagickB200Error):
        im.ResizeImage(_dev(src), 8, 8, 34)                               # SentinelFilter: not a filter
    with pytest.raises(im.MagickB200Error):
        im.AcquireKernelInfo("nosuchkernel:3")
    with pytest.raises(im.MagickB200Error):
        im.ResizeImage(_dev(src), 0, 8)


def test_magickcore_shim_end_to_end():
    """The drop-in boundary: ImageMagick's own BlurImage/ResizeImage/MorphologyImage/... entry points
    (unmodified reference library, ld --wrap) served by the GPU and compared with the stock CPU path.
    The harness is built next to the reference library (oracle/_ref/shim) where the source tree is readable and goes
    wherever oracle/_ref goes."""
    import subprocess
    exe = util.SHIM_DIR / "shim_harness"
    if not exe.exists():
        pytest.skip("shim harness not built (needs an ImageMagick source tree: IMAGEMAGICK_SOURCE=<tree> python __graft_entry__.py)")
    p = subprocess.run([str(exe)], capture_output=True, text=True, timeout=600)
    print(p.stdout)
    assert p.returncode == 0, p.stdout + p.stderr
    assert "gpu hits" in p.stdout and "FAIL" not in p.stdout
