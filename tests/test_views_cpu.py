"""tmpt_render_views without a device: the argument checks of the entry point, its declaration, and the binding's camera shapes."""
import ctypes as C
import os

import numpy as np
import pytest

import toymeshpathtracer_b200 as tm
from conftest import ROOT


def test_render_views_checks_its_arguments():
    """Each argument error returns TMPT_ERR_ARG and leaves a message, before any device work (no GPU needed)."""
    L = tm.lib()
    N = None
    fake_scene = C.create_string_buffer(4096)  # never dereferenced: every call below fails its argument checks first
    cams = (C.c_float * (22 * 4))()
    rgba = (C.c_uint8 * 64)()
    s, c = C.cast(fake_scene, C.c_void_p), C.cast(cams, C.c_void_p)
    none = tm.Outputs()
    only_rgba = tm.Outputs(rgba=C.addressof(rgba))

    def views(scene=s, cameras=c, n=4, w=4, h=4, spp=1, mem=tm.HOST, out=C.byref(only_rgba)):
        return L.tmpt_render_views(scene, cameras, n, w, h, spp, mem, out, N, N, N)

    calls = {
        "NULL scene": (lambda: views(scene=N), "NULL scene / cameras"),
        "NULL cameras": (lambda: views(cameras=N), "NULL scene / cameras"),
        "no views": (lambda: views(n=0), "nViews 0 out of range 1..65536"),
        "negative views": (lambda: views(n=-3), "nViews -3 out of range"),
        "65537 views": (lambda: views(n=65537), "nViews 65537 out of range"),
        "width 0": (lambda: views(w=0), "out of range"),
        "height 10001": (lambda: views(h=10001), "out of range"),
        "spp 0": (lambda: views(spp=0), "out of range"),
        "spp 1025": (lambda: views(spp=1025), "out of range"),
        "more than 10^8 pixels": (lambda: views(n=65536, w=40, h=40), "more than 100000000 pixels"),
        "10^8 pixels and one row": (lambda: views(n=10001, w=10000, h=1), "more than 100000000 pixels"),
        "NULL out": (lambda: views(out=N), "out is NULL"),
        "nothing requested": (lambda: views(out=C.byref(none)), "no output requested"),
        "bad mem": (lambda: views(mem=5), "mem 5"),
    }
    for name, (call, message) in calls.items():
        assert call() == tm.TMPT_ERR_ARG, name
        msg = L.tmpt_last_error().decode()
        assert message in msg, (name, msg)
        if name not in ("width 0", "height 10001", "spp 0", "spp 1025"):
            assert "tmpt_render_views" in msg, (name, msg)


def test_header_declares_render_views_at_abi_version_3():
    hdr = open(os.path.join(ROOT, "include", "tmpt.h")).read()
    assert "#define TMPT_ABI_VERSION 3" in hdr
    assert "int tmpt_render_views(const tmpt_scene* scene, const tmpt_camera* cameras, int nViews, int width, int height, int spp," in hdr
    assert "tmpt_render_views" in tm.ABI_SYMBOLS


@pytest.mark.parametrize("shape", [(22,), (3, 21), (2, 22, 1), (0, 22, 2), (4, 23)])
def test_render_views_rejects_cameras_of_the_wrong_shape(shape):
    """The binding's shape check comes before the scene is touched: a Scene without a device is never built here."""
    scene = tm.Scene.__new__(tm.Scene)  # (no handle: the ValueError must come first)
    scene._h = None
    cams = np.zeros(shape, np.float32)
    with pytest.raises(ValueError, match=r"\[N, 22\]"):
        scene.render_views(cams, 4, 4, 1)
    with pytest.raises(ValueError, match=r"\[N, 22\]"):
        scene.render_views_device(cams, 4, 4, 1, rgba_ptr=1)
