"""CPU-only checks of the product's host side (no GPU compute calls):
 * libmagickb200.so loads and exports every symbol include/magick_b200.h declares,
 * kernel builders / parser produce taps bit-identical to the reference's (golden + oracle),
 * resize contribution tables equal the oracle's weights,
 * the operators fail loudly (no CPU fallback) when there is no CUDA device."""
import ctypes as C
import re
from pathlib import Path

import numpy as np
import pytest

import util

im = pytest.importorskip("imagemagick_b200")
from imagemagick_b200 import _lib  # noqa: E402

ROOT = Path(__file__).resolve().parent.parent
G = np.load(ROOT / "tests" / "golden" / "hotpath_golden.npz")


def test_every_declared_symbol_is_exported():
    header = (ROOT / "include" / "magick_b200.h").read_text()
    declared = set(re.findall(r"\b(mb200_[a-z0-9_]+)\s*\(", header))
    declared -= {"mb200_kernel_info", "mb200_kernel_type"}      # type names mentioned in comments
    assert len(declared) >= 35
    lib = C.CDLL(str(_lib.LIB_PATH))
    missing = [s for s in sorted(declared) if not hasattr(lib, s)]
    assert not missing, missing
    assert declared == set(_lib.PROTOTYPES), declared ^ set(_lib.PROTOTYPES)
    assert b"sm_100a" in _lib.load().mb200_version()


def same_kernel(a, b):
    return a.shape == b.shape and np.array_equal(np.isnan(a), np.isnan(b)) and \
        np.array_equal(a[~np.isnan(a)].view(np.int64), b[~np.isnan(b)].view(np.int64))


@pytest.mark.parametrize("ks", [k.split("/", 1)[1] for k in G.files if k.startswith("kernel/")])
def test_kernel_strings_match_reference_taps(ks):
    vals, x, y = im.AcquireKernelInfo(ks).arrays()[0]
    assert same_kernel(vals, G["kernel/" + ks]), ks
    assert [x, y] == list(G["kernel_origin/" + ks]), ks


def test_kernel_list_and_user_arrays():
    ks = im.AcquireKernelInfo("blur:0x4;blur:0x4+90").arrays()
    assert [k[0].shape for k in ks] == [(1, 33), (33, 1)]
    assert same_kernel(ks[0][0].ravel(), ks[1][0].ravel())
    (v, x, y), = im.AcquireKernelInfo("3x3+0+2: 1,2,0.5 0,-1,nan 3,0.25,-").arrays()
    assert (x, y) == (0, 2) and np.isnan(v[1, 2]) and np.isnan(v[2, 2]) and v[2, 0] == 3
    (v, x, y), = im.AcquireKernelInfo("1,1,1,1,4,1,1,1,1").arrays()
    assert v.shape == (3, 3) and (x, y) == (1, 1) and v[1, 1] == 4
    assert len(im.AcquireKernelInfo("Disk:3>").arrays()) == 1        # a disk turned by 90 degrees is the same disk: no list
    assert len(im.AcquireKernelInfo("3>: 0,0,nan 0,1,1 nan,1,nan").arrays()) == 4
    for bad in ("nosuch:3", "3x3: 1,2,3", "", "Sobel@"):
        with pytest.raises(im.MagickB200Error):
            im.AcquireKernelInfo(bad)


@pytest.mark.parametrize("r,s", [(0, 0.5), (0, 1), (0, 2), (0, 3.3), (0, 4), (0, 8), (2, 1), (7.5, 3)])
def test_optimal_widths_and_blur_taps_match_oracle(r, s):
    lib, o = _lib.load(), util.oracle()
    assert lib.mb200_optimal_kernel_width_1d(r, s) == o.orc_optimal_kernel_width_1d(r, s)
    assert lib.mb200_optimal_kernel_width_2d(r, s) == o.orc_optimal_kernel_width_2d(r, s)
    mine = im.AcquireKernelBuiltIn(im.BlurKernel, r, s, 90.0).arrays()[0]
    want = util.orc_kernel("blur", r, s, 90.0)
    assert same_kernel(mine[0], want.array()) and (mine[1], mine[2]) == (want.x, want.y)
    mine = im.AcquireKernelBuiltIn(im.GaussianKernel, r, s).arrays()[0]
    assert same_kernel(mine[0], util.orc_kernel("gaussian", r, s).array())


@pytest.mark.parametrize("filt", list(range(1, 34)))     # every FilterType, Jinc (13) and Kaiser (16) included
def test_filter_weights_match_oracle(filt):
    lib, o = _lib.load(), util.oracle()
    assert lib.mb200_resize_filter_support(filt) == o.orc_filter_support(filt)
    for x in np.concatenate([np.linspace(-5.0, 5.0, 401), [2.5464790894703255, 2.6, 3.2383154841662362, 0.999999, 1.0]]):
        a, b = lib.mb200_resize_filter_weight(filt, float(x)), o.orc_filter_weight(filt, float(x))
        assert a == b or (np.isnan(a) and np.isnan(b)), (filt, x)


EXPERT = [(22, dict(blur=0.8)), (22, dict(lobes=2)), (22, dict(lobes=5, blur=1.1)), (8, dict(sigma=0.75)),
          (8, dict(sigma=0.3, support=1.25)), (16, dict(kaiser_beta=4.5)), (16, dict(kaiser_beta=8.0, lobes=4)), (10, dict(b=0.5)),
          (10, dict(c=0.75)), (12, dict(b=0.2, c=0.6)), (3, dict(window=5)), (22, dict(window=7, win_support=2.0)),
          (11, dict(window=17, keep_filter=1)), (13, dict(lobes=2)), (13, dict(lobes=20, blur=0.9)), (21, dict(support=3.0)),
          (14, dict(support=2.5, win_support=4.0))]


@pytest.mark.parametrize("filt,values", EXPERT)
def test_expert_filter_settings_match_oracle(filt, values):
    """The "filter:*" settings as values (mb200_filter_options): weights, support and whole contribution tables are the
    oracle's -- which is pinned to the reference with the artifacts set (test_resize_expert_settings_bit_exact)."""
    lib, o = _lib.load(), util.oracle()
    opts = util.FilterOptions.of(**values)
    ref = C.byref(opts)
    assert lib.mb200_resize_filter_support_ex(filt, ref) == o.orc_filter_support_ex(filt, ref)
    for x in np.linspace(-6.0, 6.0, 241):
        a, b = lib.mb200_resize_filter_weight_ex(filt, ref, float(x)), o.orc_filter_weight_ex(filt, ref, float(x))
        assert a == b or (np.isnan(a) and np.isnan(b)), (filt, values, x)
    # the image-level oracle and the host table builder agree on which taps exist (a 1-D image makes the table visible)
    n_in, n_out = 97, 41
    taps = lib.mb200_resize_contributions_ex(filt, ref, n_in, n_out, n_out / n_in, None, None, None, 0)
    assert taps > 0
    start, count = (C.c_long * n_out)(), (C.c_int * n_out)()
    w = (C.c_double * (n_out * taps))()
    assert lib.mb200_resize_contributions_ex(filt, ref, n_in, n_out, n_out / n_in, start, count, w, taps) == taps
    w = np.array(w).reshape(n_out, taps)
    src = util.make_image(n_in, 1, 1, seed=3)
    want = np.empty((1, n_out, 1), np.float32)
    assert o.orc_resize_ex(util.P(src), n_in, 1, 1, util.P(want), n_out, 1, filt, ref) == 0
    line = src[0, :, 0].astype(np.float64)
    got = np.array([np.float32(sum(w[k, j] * line[start[k] + j] for j in range(count[k]))) for k in range(n_out)], np.float32)
    assert util.max_ulp(got.reshape(1, n_out, 1), want) <= 1


@pytest.mark.parametrize("values", [dict(), dict(film_gamma=0.5, reference_black=64.0, reference_white=940.0),
                                    dict(film_gamma=0.65, reference_white=700.0), dict(reference_black=0.0, reference_white=1024.0),
                                    dict(film_gamma=0.0)])
def test_log_and_ycc_tables_match_oracle(values):
    """The host-built tables behind the Log and YCC colourspace legs are the oracle's bit for bit (the oracle is pinned to the
    reference with the properties set, test_colorspace_settings_bit_exact), and the python mirror parses the image settings
    into the same values the tests pass directly."""
    import imagemagick_b200 as im
    lib, o = _lib.load(), util.oracle()
    opts = util.ColorspaceOptions.of(**values)
    for forward in (1, 0):
        a, b = np.empty(65536, np.float32), np.empty(65536, np.float32)
        assert lib.mb200_log_colorspace_table(forward, C.byref(opts), a.ctypes.data) == 0
        o.orc_log_table(forward, C.byref(opts), util.P(b))
        assert np.array_equal(np.isnan(a), np.isnan(b)) and np.array_equal(np.nan_to_num(a), np.nan_to_num(b)), (forward, values)
    a, b = np.empty(1389, np.float32), np.empty(1389, np.float32)
    assert lib.mb200_ycc_table(a.ctypes.data) == 0
    o.orc_ycc_table(util.P(b))
    assert np.array_equal(a, b) and a[0] == 0.0 and a[-1] == 1.0 and np.all(np.diff(a) > 0)
    names = {"film_gamma": "film-gamma", "reference_black": "reference-black", "reference_white": "reference-white"}
    parsed = im.api.colorspace_options_from_settings({names[k]: repr(v) for k, v in values.items()})
    if values:
        assert parsed.set == opts.set
        assert all(getattr(parsed, k) == getattr(opts, k) for k in values)
    else:
        assert parsed is None
    ill = im.api.colorspace_options_from_settings({"color:illuminant": "d50", "white-luminance": "203"})
    assert (ill.set, ill.illuminant, ill.white_luminance) == (3, 3, 203.0)
    assert im.api.colorspace_options_from_settings({"color:illuminant": "nonsense"}).illuminant == 5


def test_resize_contributions_lanczos_2x():
    lib = _lib.load()
    n_in, n_out = 64, 32
    taps = lib.mb200_resize_contributions(22, n_in, n_out, 0.5, None, None, None, 0)
    assert taps == 15                                   # (size_t)(2*6+3), resize.c:3379
    start = (C.c_long * n_out)()
    count = (C.c_int * n_out)()
    w = (C.c_double * (n_out * taps))()
    assert lib.mb200_resize_contributions(22, n_in, n_out, 0.5, start, count, w, taps) == taps
    w = np.array(w).reshape(n_out, taps)
    assert max(count) == 12 and count[10] == 12 and start[10] == 2 * 10 - 5
    assert np.allclose(w.sum(1), 1.0, atol=1e-14)
    # an interior row reproduces the reference's weights: normalised Lanczos3 at half-pixel phase
    o = util.oracle()
    scale = 1.0 / (1.0 / 0.5 + 1e-12)                   # resize.c:3363, :3386
    raw = np.array([o.orc_filter_weight(22, scale * ((start[10] + j) - ((10 + 0.5) / 0.5 + 1e-12) + 0.5)) for j in range(12)])
    assert np.allclose(w[10, :12], raw * (1.0 / raw.sum()), rtol=0, atol=1e-16)
    assert lib.mb200_resize_contributions(13, n_in, n_out, 0.5, None, None, None, 0) == 15   # Jinc: support 3.238.. * 2 -> 2*6.48+3
    assert lib.mb200_resize_contributions(0, n_in, n_out, 0.5, None, None, None, 0) == _lib.EUNSUPPORTED  # Undefined


def test_no_gpu_means_loud_failure_not_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    src = util.make_image(8, 8, 4)
    with pytest.raises(im.MagickB200Error) as e:
        im.BlurImage(im.Image(src), 0, 2)
    assert e.value.code == _lib.ENODEVICE
    with pytest.raises(im.MagickB200Error):
        im.ResizeImage(im.Image(src), 4, 4, im.LanczosFilter)
    assert _lib.load().mb200_device_count() == 0


def test_bench_reference_arm_contract():
    """`bench.py --impl reference` (the CPU arm the driver runs next to the GPU arm): one JSON line with the
    contract's keys; it times the real reference (oracle/_ref) when that library exists, else the oracle port."""
    import json
    import subprocess
    import sys
    env = dict(**__import__("os").environ, OMP_NUM_THREADS="", MB200_BENCH_CPU_SIZE="1024")
    p = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=600, env=env)
    assert p.returncode == 0, p.stderr[-500:]
    line = json.loads([l for l in p.stdout.splitlines() if l.startswith("{")][-1])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
                "scaling", "dtype", "data", "config", "cpu_baseline", "e2e", "gpu_launches"):
        assert key in line, key
    assert line["impl"] == "reference" and line["unit"] == "Mpixels/s" and line["value"] > 0
    assert line["cpu_baseline"]["kind"] in ("reference", "port") and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0
    assert "workload" in line["config"] and "8192x8192" in line["config"]["workload"]
    assert "1024x1024" in line["cpu_baseline"]["sample"]          # this test shrinks the sample; the driver runs 8192^2


def test_sharpen_and_edge_kernels_match_the_reference_taps():
    """effect.c:3991 / :1520 build their kernels inline; convolving a one-pixel impulse with the real
    SharpenImage / EdgeImage returns those taps (reflected), which must equal the product's host-built kernels."""
    lib = _lib.load()
    for name, build, ref_call in (
            ("sharpen", lambda: lib.mb200_sharpen_kernel(0.0, 1.0), lambda s, n: util.ref_output("ref_sharpen", s, util.OUT, n, n, 1, 0.0, 1.0, shape=s.shape)),
            ("sharpen r2", lambda: lib.mb200_sharpen_kernel(2.0, 0.7), lambda s, n: util.ref_output("ref_sharpen", s, util.OUT, n, n, 1, 2.0, 0.7, shape=s.shape)),
            ("edge", lambda: lib.mb200_edge_kernel(1.0), lambda s, n: util.ref_output("ref_edge", s, util.OUT, n, n, 1, 1.0, shape=s.shape))):
        k = im.KernelInfo(build())
        vals, kx, ky = k.arrays()[0]
        w = vals.shape[0]
        n = w + 8
        src = np.zeros((n, n, 1), np.float32)
        src[n // 2, n // 2, 0] = 1.0
        dst = ref_call(src, n)
        got = dst[n // 2 - ky: n // 2 - ky + w, n // 2 - kx: n // 2 - kx + w, 0]
        want = vals[::-1, ::-1].astype(np.float32)          # convolution reflects the kernel
        assert np.array_equal(got, want), name


def test_threshold_geometry_is_parsed_before_the_device_is_touched():
    """Black/WhiteThreshold: syntax the host parser does not take and images the reference first promotes
    (gray) or gamma-encodes (linear RGB) are declined (EUNSUPPORTED) -- decided on the host, GPU or not."""
    lib = _lib.load()
    buf = np.zeros((4, 4, 4), np.float32)
    for bad in (b"50%x20", b"a,b", b"1,2,3,4,5", b""):
        assert lib.mb200_black_threshold_image_dev(buf.ctypes.data, 4, 4, 4, 23, bad, None) == _lib.EUNSUPPORTED
    assert lib.mb200_white_threshold_image_dev(buf.ctypes.data, 4, 4, 2, 23, b"50%", None) == _lib.EUNSUPPORTED   # gray+alpha
    assert lib.mb200_white_threshold_image_dev(buf.ctypes.data, 4, 4, 4, 21, b"50%", None) == _lib.EUNSUPPORTED   # linear RGB
    if lib.mb200_device_count() == 0:                            # (never hand a host pointer to a real device)
        rc = lib.mb200_black_threshold_image_dev(buf.ctypes.data, 4, 4, 4, 23, b"10%,20%,30%", None)
        assert rc in (_lib.ENODEVICE, _lib.ECUDA)                # well-formed: only the missing device stops it


def test_header_is_plain_c99_and_links(tmp_path):
    """The boundary is a C ABI: include/magick_b200.h compiles as strict C99 (no C++-isms, no CUDA types) and
    examples/blur_resize.c links against the shared library and runs (it stops after printing the version when
    there is no device)."""
    import shutil
    import subprocess
    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("no gcc")
    exe = tmp_path / "blur_resize"
    libdir = _lib.LIB_PATH.parent
    subprocess.run([gcc, "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", f"-I{ROOT / 'include'}",
                    str(ROOT / "examples" / "blur_resize.c"), f"-L{libdir}", "-lmagickb200", f"-Wl,-rpath,{libdir}",
                    "-o", str(exe)], check=True, capture_output=True)
    if _lib.load().mb200_device_count() == 0:
        p = subprocess.run([str(exe), "64", "64"], capture_output=True, text=True, timeout=120)
        assert p.returncode == 0 and "sm_100a" in p.stdout


def test_process_filter_module_on_the_cpu_path():
    """imagemagick_b200/shim/b200_filter.c (`magick ... -process "b200 blur 0x2 resize 50% ..."`): driven like
    InvokeDynamicImageFilter on a two-image list.  Without a device every accelerate call declines, so the filter
    must reproduce the stock operators bit for bit, keep the list intact and reject unknown operators."""
    import os
    import subprocess
    exe = util.SHIM_DIR / "filter_harness"
    if not exe.exists():
        pytest.skip("filter_harness not built (needs an ImageMagick source tree: IMAGEMAGICK_SOURCE=<tree> python __graft_entry__.py)")
    env = dict(os.environ)
    if _lib.load().mb200_device_count() == 0:
        env["B200_FILTER_EXPECT_EXACT"] = "1"
    p = subprocess.run([str(exe)], capture_output=True, text=True, timeout=300, env=env)
    assert p.returncode == 0, p.stdout + p.stderr
    assert "ok" in p.stdout


def test_wrapped_entry_points_fall_back_on_the_cpu():
    """shim_harness (ld --wrap build of the unmodified reference) without a device: every wrapped entry point
    declines silently and returns exactly what the stock function returns -- including __wrap_ThumbnailImage,
    whose cascade is re-issued by the shim and whose Thumb::* metadata comes from the real function."""
    import subprocess
    exe = util.SHIM_DIR / "shim_harness"
    if not exe.exists():
        pytest.skip("shim_harness not built (needs an ImageMagick source tree: IMAGEMAGICK_SOURCE=<tree> python __graft_entry__.py)")
    if _lib.load().mb200_device_count() != 0:
        pytest.skip("device present: the GPU variant of this check is tests/test_gpu_parity.py::test_magickcore_shim_end_to_end")
    p = subprocess.run([str(exe)], capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-500:]
    assert "FAIL" not in p.stdout and "gpu hits 0" in p.stdout
    assert p.stdout.count("ThumbnailImage RGBA") == 3


@pytest.mark.parametrize("rad,sig,ang", [(0, 2, 0), (0, 2, 45), (0, 3, 90), (0, 1.5, -30), (0, 4, 180), (5, 2, 270), (0, 2, 123.4)])
def test_motion_blur_taps_and_offsets_match_the_reference(rad, sig, ang):
    """The product builds MotionBlurImage's taps / offsets on the host (effect.c:2316-2345, :2390-2398); the real
    MotionBlurImage applied to a one-pixel impulse scatters exactly those taps to -offset."""
    lib = _lib.load()
    n = lib.mb200_motion_blur_kernel(rad, sig, ang, None, None, None, 0)
    t, ox, oy = (C.c_double * n)(), (C.c_long * n)(), (C.c_long * n)()
    assert lib.mb200_motion_blur_kernel(rad, sig, ang, t, ox, oy, n) == n
    size = 2 * n + 5
    c = size // 2
    src = np.zeros((size, size, 1), np.float32)
    src[c, c, 0] = 1.0
    want = np.zeros((size, size), np.float64)
    for j in range(n):                      # out[y][x] = sum_j k_j * src[y + oy_j][x + ox_j], accumulated in tap order
        want[c - oy[j], c - ox[j]] += t[j]
    util.expect_ref(want.astype(np.float32)[..., None], "ref_motion_blur", src, util.OUT, size, size, 1, rad, sig, ang)


@pytest.mark.parametrize("sizes", [((37, 23), (19, 11)), ((20, 14), (53, 31)), ((31, 17), (31, 9)), ((64, 8), (21, 8))])
def test_scale_contribution_lists_reproduce_the_oracle(sizes):
    """ScaleImage's term lists are host logic (resize_filter.cpp mb200_scale_contributions): folding them in float64 --
    acc = acc + w * v, the arithmetic the gather kernel performs -- must reproduce the oracle's literal restatement of
    the reference's state machine bit for bit (the oracle itself is pinned to the compiled reference)."""
    (w, h), (ow, oh) = sizes
    lib = _lib.load()
    src = util.make_image(w, h, 3, seed=12)

    def lists(axis, n_in, n_out):
        off = (C.c_long * (n_out + 1))()
        total = lib.mb200_scale_contributions(axis, n_in, n_out, off, None, None, 0)
        assert total > 0
        idx, wt = (C.c_int * total)(), (C.c_double * total)()
        assert lib.mb200_scale_contributions(axis, n_in, n_out, off, idx, wt, total) == total
        return list(off), list(idx), list(wt)

    xo, xi, xw = lists(0, w, ow)
    yo, yi, yw = lists(1, h, oh)
    got = np.empty((oh, ow, 3), np.float32)
    s64 = src.astype(np.float64)
    for y in range(oh):
        for t in range(ow):
            pixel = np.zeros(3)
            for j in range(xo[t], xo[t + 1]):
                col = np.zeros(3)
                for k in range(yo[y], yo[y + 1]):
                    col = col + yw[k] * s64[yi[k], xi[j]]
                pixel = pixel + xw[j] * col
            got[y, t] = pixel.astype(np.float32)
    want = np.empty((oh, ow, 3), np.float32)
    assert util.oracle().orc_scale(util.P(src), w, h, 3, util.P(want), ow, oh) == 0
    assert np.array_equal(got, want)
