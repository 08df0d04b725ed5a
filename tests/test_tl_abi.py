"""CPU tests of the tangent-linear entry points (include/paradis_sl_tl.h): every declared function is exported and
bound by its own ctypes table, and bad arguments are rejected with the documented codes before a GPU is touched."""
import ctypes as C
import os
import re

from conftest import ROOT
from paradis_model_b200 import _lib, build


def tl_header_functions():
    text = open(os.path.join(ROOT, "include", "paradis_sl_tl.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(paradis_[a-z0-9_]+)\s*\(", text)))


def test_tl_header_exported_and_bound():
    names = tl_header_functions()
    assert names == ["paradis_sl_advect_jvp", "paradis_sl_advect_jvp_workspace"]
    handle = C.CDLL(build.build_library())
    for n in names:
        assert hasattr(handle, n), f"{n} declared in include/paradis_sl_tl.h but not exported"
    assert sorted(_lib.exported_symbols_tl()) == names
    for other in (_lib.exported_symbols(), _lib.exported_symbols_bf16(), _lib.exported_symbols_geocyclic()):
        assert not set(names) & set(other)
    assert _lib.lib().paradis_sl_abi_version() == 2
    assert os.path.join(ROOT, "paradis_model_b200", "..", "include", "paradis_sl_tl.h") in build.HEADERS


def _geom(H=8, W=16):
    g = _lib.Geom()
    g.H, g.W = H, W
    g.sin_lat = g.cos_lat = g.lon = 256          # non-NULL dummies, never dereferenced on the host
    g.own_rows = g.arr_rows = g.fld_rows = H
    return g


def _jvp(g, field, dfield, u, v, du, dv, dout, interp=1, pole_fix=1, ws=None, ws_bytes=0):
    sB = 128
    return _lib.lib().paradis_sl_advect_jvp(C.byref(g), field, dfield, u, v, du, dv, dout, 1, 1, sB, sB, sB, sB, sB,
                                            sB, 0.1, interp, pole_fix, 0, ws, ws_bytes, None, None)


def test_tl_argument_errors_without_gpu():
    L = _lib.lib()
    a = C.c_void_p(4096)
    ws = C.c_void_p(1 << 20)
    nb = L.paradis_sl_advect_jvp_workspace(1, 1)
    assert nb >= 2 * L.paradis_sl_advect_fwd_workspace(1, 1)      # pole means of field and of dfield
    ok = dict(ws=ws, ws_bytes=nb)
    # bad interpolation: the forward's code
    assert _jvp(_geom(), a, a, a, a, a, a, a, interp=3, **ok) == 3
    assert _jvp(_geom(), a, a, a, a, a, a, a, interp=0, **ok) == 3
    # NULL field / u / v / dout
    assert _jvp(_geom(), None, a, a, a, a, a, a, **ok) == 4
    assert _jvp(_geom(), a, a, None, a, a, a, a, **ok) == 4
    assert _jvp(_geom(), a, a, a, None, a, a, a, **ok) == 4
    assert _jvp(_geom(), a, a, a, a, a, a, None, **ok) == 4
    # only one of du / dv
    assert _jvp(_geom(), a, a, a, a, a, None, a, **ok) == 4 and b"du and dv" in L.paradis_last_error()
    assert _jvp(_geom(), a, a, a, a, None, a, a, **ok) == 4
    # latitude-band windows and peer halos
    g = _geom(); g.own_row0, g.own_rows = 2, 4
    assert _jvp(g, a, a, a, a, a, a, a, **ok) == 1 and b"full mesh" in L.paradis_last_error()
    g = _geom(); g.fld_row0, g.fld_rows = 1, 6
    assert _jvp(g, a, a, a, a, a, a, a, **ok) == 1
    g = _geom(); g.fld_peer_lo, g.fld_peer_rows = 4096, 2
    assert _jvp(g, a, a, a, a, a, a, a, **ok) == 1 and b"peer" in L.paradis_last_error()
    # shape errors of the forward
    assert _jvp(_geom(8, 15), a, a, a, a, a, a, a, **ok) == 2
    assert _jvp(_geom(0, 16), a, a, a, a, a, a, a, **ok) == 1
    # workspace too small (every other argument valid: the next step would be a launch); none needed without pole_fix
    assert _jvp(_geom(), a, a, a, a, a, a, a, ws=None, ws_bytes=0) == 5
    assert _jvp(_geom(), a, a, a, a, a, a, a, ws=ws, ws_bytes=nb - 1) == 5
    assert _jvp(_geom(), a, None, a, a, a, a, a, ws=None, ws_bytes=0) == 5
