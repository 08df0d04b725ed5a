"""CPU tests of include/paradis_geocyclic.h (bf16 storage of the GeoCyclic pad / depthwise-convolution / avgpool5 ops
and the avgpool5 adjoint): every declared function is exported and bound by the third ctypes table, and bad arguments
are rejected with the documented codes before a GPU is touched."""
import ctypes as C
import os
import re

from conftest import ROOT
from paradis_model_b200 import _lib, build

HEADER = os.path.join(ROOT, "include", "paradis_geocyclic.h")


def header_functions():
    text = re.sub(r"/\*.*?\*/", "", open(HEADER).read(), flags=re.S)
    return sorted(set(re.findall(r"\b(paradis_[a-z0-9_]+)\s*\(", text)))


def test_geocyclic_header_exported_and_bound():
    names = header_functions()
    assert names == sorted([
        "paradis_geocyclic_pad_fwd_bf16", "paradis_geocyclic_pad_bwd_bf16",
        "paradis_geocyclic_dwconv_fwd_bf16", "paradis_geocyclic_dwconv_bwd_input_bf16",
        "paradis_geocyclic_dwconv_bwd_weight_bf16",
        "paradis_geocyclic_avgpool5_fwd_bf16", "paradis_geocyclic_avgpool5_bwd", "paradis_geocyclic_avgpool5_bwd_bf16"])
    handle = C.CDLL(build.build_library())
    for n in names:
        assert hasattr(handle, n), f"{n} declared in include/paradis_geocyclic.h but not exported"
    assert sorted(_lib.exported_symbols_geocyclic()) == names
    assert not set(names) & set(_lib.exported_symbols())
    assert not set(names) & set(_lib.exported_symbols_bf16())
    assert _lib.lib().paradis_sl_abi_version() == 2
    assert os.path.join(ROOT, "paradis_model_b200", "..", "include", "paradis_geocyclic.h") in build.HEADERS


A = C.c_void_p(4096)            # aligned dummy device pointers, never dereferenced on the host
WS = C.c_void_p(1 << 20)


def _dw(name, B=1, Cn=2, H=12, W=16, k=3, x=A, y=A, weight=A, ws_bytes=None):
    L = _lib.lib()
    if name == "fwd":
        return L.paradis_geocyclic_dwconv_fwd_bf16(x, weight, None, y, B, Cn, H, W, k, None)
    if name == "bwd_input":
        return L.paradis_geocyclic_dwconv_bwd_input_bf16(x, weight, y, B, Cn, H, W, k, None)
    if ws_bytes is None:
        ws_bytes = L.paradis_geocyclic_dwconv_wgrad_workspace(B, Cn, H, W, k)
    return L.paradis_geocyclic_dwconv_bwd_weight_bf16(x, y, weight, None, B, Cn, H, W, k, WS, ws_bytes, None)


def _pool(name, B=1, Cn=2, H=12, W=16, stride=2, x=A, y=A):
    return getattr(_lib.lib(), name)(x, y, B, Cn, H, W, stride, None)


POOLS = ["paradis_geocyclic_avgpool5_fwd_bf16", "paradis_geocyclic_avgpool5_bwd", "paradis_geocyclic_avgpool5_bwd_bf16"]
PADS = ["paradis_geocyclic_pad_fwd_bf16", "paradis_geocyclic_pad_bwd_bf16"]


def test_geocyclic_argument_errors_without_gpu():
    L = _lib.lib()
    for name in ("fwd", "bwd_input", "bwd_weight"):
        assert _dw(name, x=None) == 4, name                       # NULL tensor
        assert _dw(name, y=None) == 4, name
        assert _dw(name, weight=None) == 4, name                  # NULL weight / grad weight
        assert _dw(name, W=15) == 2, name                          # odd W
        assert _dw(name, k=4) == 3 and _dw(name, k=9) == 3, name   # k not in {3, 5, 7}
        assert _dw(name, H=5, k=5) == 1, name                      # H < k + 1
        assert _dw(name, W=4, k=7) == 1, name                      # W < k - 1
        assert _dw(name, B=2, Cn=40000) == 1, name                 # B * C > 65535
    assert _dw("bwd_weight", ws_bytes=L.paradis_geocyclic_dwconv_wgrad_workspace(1, 2, 12, 16, 3) - 4) == 5
    assert b"workspace" in L.paradis_last_error()
    for name in POOLS:
        assert _pool(name, x=None) == 4 and _pool(name, y=None) == 4, name
        assert _pool(name, W=15) == 2, name
        assert _pool(name, H=5) == 1, name                         # the 5x5 window needs H >= 6
        assert _pool(name, B=300, Cn=300) == 1, name
        assert _pool(name, stride=0) == 1 and b"stride" in L.paradis_last_error(), name
    for name in PADS:
        fn = getattr(L, name)
        assert fn(None, A, 2, 8, 16, 1, None) == 4 and fn(A, None, 2, 8, 16, 1, None) == 4, name
        assert fn(A, A, 2, 8, 15, 1, None) == 2, name              # odd W
        assert fn(A, A, 2, 2, 16, 3, None) == 1, name              # H < p + 1
        assert fn(A, A, 70000, 8, 16, 1, None) == 1, name          # planes > 65535
    misaligned = C.c_void_p(4096 + 2)                              # the forward stores two values per 4-byte word
    assert L.paradis_geocyclic_pad_fwd_bf16(A, misaligned, 2, 8, 16, 1, None) == 1
    assert b"aligned" in L.paradis_last_error()
