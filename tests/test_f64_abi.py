"""CPU tests of the float64 entry points (include/paradis_sl_f64.h): every declared function is exported and bound by
its own ctypes table, and bad arguments are rejected with the documented codes before a GPU is touched."""
import ctypes as C
import os
import re

from conftest import ROOT
from paradis_model_b200 import _lib, build


def f64_header_functions():
    text = open(os.path.join(ROOT, "include", "paradis_sl_f64.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(paradis_[a-z0-9_]+)\s*\(", text)))


def test_f64_header_exported_and_bound():
    names = f64_header_functions()
    assert len(names) == 15 and all("f64" in n for n in names)
    handle = C.CDLL(build.build_library())
    for n in names:
        assert hasattr(handle, n), f"{n} declared in include/paradis_sl_f64.h but not exported"
    assert sorted(_lib.exported_symbols_f64()) == names
    for other in (_lib.exported_symbols(), _lib.exported_symbols_bf16(), _lib.exported_symbols_geocyclic(),
                  _lib.exported_symbols_tl()):
        assert not set(names) & set(other)
    assert _lib.lib().paradis_sl_abi_version() == 2
    assert os.path.join(ROOT, "paradis_model_b200", "..", "include", "paradis_sl_f64.h") in build.HEADERS


def _geom(H=8, W=16):
    g = _lib.GeomF64()
    g.H, g.W = H, W
    g.sin_lat = g.cos_lat = g.lon = 256          # non-NULL dummies, never dereferenced on the host
    g.min_lat, g.d_lat, g.min_lon, g.d_lon = -1.5, 3.0, 0.0, 6.0
    return g


A = C.c_void_p(4096)
WS = C.c_void_p(1 << 20)


def _fwd(g, field=A, u=A, v=A, out=A, interp=1, pole_fix=1, ws=WS, ws_bytes=1 << 20):
    return _lib.lib().paradis_sl_advect_fwd_f64(C.byref(g), field, u, v, out, 1, 1, 128, 128, 128, 0.1, interp,
                                                pole_fix, 0, ws, ws_bytes, None, None)


def _bwd(g, gout=A, field=A, u=A, v=A, gf=A, gu=A, gv=A, interp=1, ws=WS, ws_bytes=None):
    L = _lib.lib()
    if ws_bytes is None:
        ws_bytes = L.paradis_sl_advect_bwd_f64_workspace(1, 1, g.H, g.W)
    return L.paradis_sl_advect_bwd_f64(C.byref(g), gout, field, u, v, gf, gu, gv, 1, 1, 128, 128, 128, 128, 0.1,
                                       interp, 1, 0, ws, ws_bytes, None, None)


def _jvp(g, field=A, dfield=A, u=A, v=A, du=A, dv=A, dout=A, interp=1, ws=WS, ws_bytes=1 << 20):
    return _lib.lib().paradis_sl_advect_jvp_f64(C.byref(g), field, dfield, u, v, du, dv, dout, 1, 1, 128, 128, 128,
                                                128, 128, 128, 0.1, interp, 1, 0, ws, ws_bytes, None, None)


def test_f64_advection_argument_errors_without_gpu():
    L = _lib.lib()
    # NULL tensors and tables
    assert _fwd(_geom(), field=None) == 4 and _fwd(_geom(), out=None) == 4
    g = _geom(); g.sin_lat = None
    assert _fwd(g) == 4
    assert _bwd(_geom(), gout=None) == 4 and _bwd(_geom(), v=None) == 4
    assert _bwd(_geom(), gu=None) == 4 and b"grad_u and grad_v" in L.paradis_last_error()
    assert _jvp(_geom(), dout=None) == 4 and _jvp(_geom(), dv=None) == 4
    assert L.paradis_sl_departure_coords_f64(C.byref(_geom()), A, None, A, 1, 1, 128, 128, 0.1, 1, 0, None) == 4
    # odd W, bad interpolation, H < p + 2
    assert _fwd(_geom(8, 15)) == 2 and _bwd(_geom(8, 15)) == 2 and _jvp(_geom(8, 15)) == 2
    assert _fwd(_geom(), interp=3) == 3 and _bwd(_geom(), interp=0) == 3 and _jvp(_geom(), interp=3) == 3
    assert _fwd(_geom(2, 16), interp=1) == 1 and _fwd(_geom(3, 16), interp=2) == 1 and _jvp(_geom(3, 16), interp=2) == 1
    # workspace too small (every other argument valid: the next step would be a launch)
    assert _fwd(_geom(), ws=None, ws_bytes=0) == 5
    assert _fwd(_geom(), ws_bytes=L.paradis_sl_advect_fwd_f64_workspace(1, 1) - 1) == 5
    assert _bwd(_geom(), ws_bytes=L.paradis_sl_advect_bwd_f64_workspace(1, 1, 8, 16) - 1) == 5
    assert _jvp(_geom(), ws_bytes=L.paradis_sl_advect_jvp_f64_workspace(1, 1) - 1) == 5
    assert L.paradis_sl_advect_jvp_f64_workspace(1, 1) >= 2 * L.paradis_sl_advect_fwd_f64_workspace(1, 1)
    # the gather's double accumulator rows: W = 1440 fits the shared memory, W = 4000 does not
    assert _bwd(_geom(8, 4000)) == 1 and b"shared memory" in L.paradis_last_error()


def test_f64_geocyclic_argument_errors_without_gpu():
    L = _lib.lib()
    assert L.paradis_geocyclic_pad_fwd_f64(None, A, 1, 8, 16, 1, None) == 4
    assert L.paradis_geocyclic_pad_bwd_f64(A, A, 1, 8, 15, 1, None) == 2
    assert L.paradis_geocyclic_pad_fwd_f64(A, A, 1, 2, 16, 2, None) == 1
    assert L.paradis_geocyclic_dwconv_fwd_f64(A, None, None, A, 1, 1, 8, 16, 3, None) == 4
    assert L.paradis_geocyclic_dwconv_fwd_f64(A, A, None, A, 1, 1, 8, 16, 4, None) == 3
    assert L.paradis_geocyclic_dwconv_bwd_input_f64(A, A, A, 1, 1, 8, 17, 3, None) == 2
    assert L.paradis_geocyclic_dwconv_bwd_input_f64(A, A, A, 1, 1, 5, 16, 5, None) == 1
    nb = L.paradis_geocyclic_dwconv_wgrad_f64_workspace(2, 3, 33, 64, 5)
    assert nb > 0
    assert L.paradis_geocyclic_dwconv_bwd_weight_f64(A, A, A, None, 2, 3, 33, 64, 5, WS, nb - 1, None) == 5
    assert L.paradis_geocyclic_dwconv_bwd_weight_f64(A, A, None, None, 2, 3, 33, 64, 5, WS, nb, None) == 4
    assert L.paradis_geocyclic_avgpool5_fwd_f64(A, A, 1, 1, 8, 16, 0, None) == 1
    assert L.paradis_geocyclic_avgpool5_bwd_f64(None, A, 1, 1, 8, 16, 2, None) == 4
