"""CPU tests of the bf16 entry points (include/paradis_sl_bf16.h): every declared function is exported and bound
by the second ctypes table, and bad arguments are rejected with the documented codes before a GPU is touched."""
import ctypes as C
import os
import re

from conftest import ROOT
from paradis_model_b200 import _lib, build


def bf16_header_functions():
    text = open(os.path.join(ROOT, "include", "paradis_sl_bf16.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(paradis_[a-z0-9_]+)\s*\(", text)))


def test_bf16_header_exported_and_bound():
    names = bf16_header_functions()
    assert names == ["paradis_sl_advect_bwd_bf16", "paradis_sl_advect_bwd_bf16_workspace", "paradis_sl_advect_fwd_bf16"]
    handle = C.CDLL(build.build_library())
    for n in names:
        assert hasattr(handle, n), f"{n} declared in include/paradis_sl_bf16.h but not exported"
    assert sorted(_lib.exported_symbols_bf16()) == names
    assert not set(names) & set(_lib.exported_symbols())          # exported_symbols() stays paradis_sl.h
    assert _lib.lib().paradis_sl_abi_version() == 2
    assert os.path.join(ROOT, "paradis_model_b200", "..", "include", "paradis_sl_bf16.h") in build.HEADERS


def _geom(H=8, W=16):
    g = _lib.Geom()
    g.H, g.W = H, W
    g.sin_lat = g.cos_lat = g.lon = 256          # non-NULL, 16-byte aligned dummies, never dereferenced on the host
    g.own_rows = g.arr_rows = g.fld_rows = H
    return g


def _fwd(g, field, u, v, out, sB=128, interp=1, pole_fix=1, ws=None, ws_bytes=0):
    return _lib.lib().paradis_sl_advect_fwd_bf16(C.byref(g), field, u, v, out, 1, 1, sB, sB, sB, 0.1, interp, pole_fix,
                                                 0, ws, ws_bytes, None, None)


def _bwd(g, ptrs, sB=128, gsB=128, interp=1, ws=None, ws_bytes=0):
    go, f, u, v, gf, gu, gv = ptrs
    return _lib.lib().paradis_sl_advect_bwd_bf16(C.byref(g), go, f, u, v, gf, gu, gv, 1, 1, gsB, sB, sB, sB, 0.1,
                                                 interp, 1, 0, 3, 8.0, ws, ws_bytes, None, None)


def test_bf16_argument_errors_without_gpu():
    L = _lib.lib()
    a = C.c_void_p(4096)                          # 16-byte aligned dummy device pointer
    odd = C.c_void_p(4096 + 8)                    # 8-byte aligned only
    ws = C.c_void_p(1 << 20)
    fwd_ws = L.paradis_sl_advect_fwd_workspace(1, 1)
    bwd_ws = L.paradis_sl_advect_bwd_bf16_workspace(1, 1, 8, 16)
    # the bf16 workspace adds the fp32 grad_field accumulation buffer to the fp32 one
    assert bwd_ws >= L.paradis_sl_advect_bwd_workspace(1, 1, 8, 16) + 8 * 16 * 4
    six = [a] * 7

    # bad interpolation
    assert _fwd(_geom(), a, a, a, a, interp=3, ws=ws, ws_bytes=fwd_ws) == 3
    assert _bwd(_geom(), six, interp=0, ws=ws, ws_bytes=bwd_ws) == 3
    # NULL tensors
    assert _fwd(_geom(), None, a, a, a, ws=ws, ws_bytes=fwd_ws) == 4
    assert _bwd(_geom(), [a, a, None, a, a, a, a], ws=ws, ws_bytes=bwd_ws) == 4
    assert _bwd(_geom(), [a, a, a, a, a, a, None], ws=ws, ws_bytes=bwd_ws) == 4      # grad_u without grad_v
    # latitude-band windows
    g = _geom(); g.own_row0, g.own_rows = 2, 4
    assert _fwd(g, a, a, a, a, ws=ws, ws_bytes=fwd_ws) == 1 and b"full mesh" in L.paradis_last_error()
    g = _geom(); g.fld_row0, g.fld_rows = 1, 6
    assert _bwd(g, six, ws=ws, ws_bytes=bwd_ws) == 1 and b"full mesh" in L.paradis_last_error()
    # peer halo pointers
    g = _geom(); g.fld_peer_lo, g.fld_peer_rows = 4096, 2
    assert _fwd(g, a, a, a, a, ws=ws, ws_bytes=fwd_ws) == 1 and b"peer" in L.paradis_last_error()
    g = _geom(); g.arr_peer_rows = 2
    for k in range(3):
        g.arr_peer_hi[k] = 4096
    assert _bwd(g, six, ws=ws, ws_bytes=bwd_ws) == 1 and b"peer" in L.paradis_last_error()
    # W % 8 != 0 (even W, so not the odd-width code)
    assert _fwd(_geom(8, 12), a, a, a, a, sB=96, ws=ws, ws_bytes=fwd_ws) == 1 and b"W % 8" in L.paradis_last_error()
    assert _bwd(_geom(8, 12), six, sB=96, gsB=96, ws=ws, ws_bytes=bwd_ws) == 1
    # misaligned pointers and batch strides
    assert _fwd(_geom(), a, odd, a, a, ws=ws, ws_bytes=fwd_ws) == 1 and b"aligned" in L.paradis_last_error()
    assert _fwd(_geom(), a, a, a, odd, ws=ws, ws_bytes=fwd_ws) == 1
    assert _bwd(_geom(), [a, a, a, a, odd, a, a], ws=ws, ws_bytes=bwd_ws) == 1
    assert _fwd(_geom(), a, a, a, a, sB=132, ws=ws, ws_bytes=fwd_ws) == 1 and b"multiples of 8" in L.paradis_last_error()
    assert _bwd(_geom(), six, gsB=130, ws=ws, ws_bytes=bwd_ws) == 1 and b"multiples of 4" in L.paradis_last_error()
    # workspace too small (every other argument is valid: the next step would be a launch)
    assert _fwd(_geom(), a, a, a, a, ws=None, ws_bytes=0) == 5
    assert _bwd(_geom(), six, ws=ws, ws_bytes=L.paradis_sl_advect_bwd_workspace(1, 1, 8, 16)) == 5
