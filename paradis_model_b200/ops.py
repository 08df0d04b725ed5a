"""torch.library custom ops over the C ABI (include/paradis_sl.h).

Ops (namespace ``paradis``)
    sl_advect / sl_advect_backward      model/advection.py:129-169, fused
    sl_advect_jvp                        its tangent-linear model (forward-mode AD), fused
    geocyclic_pad / geocyclic_pad_backward   model/padding.py:11-39
    geocyclic_dwconv / geocyclic_dwconv_backward(_bf16)   SepConv's pad + depthwise conv, model/blocks.py:112-114
    geocyclic_avgpool5 / geocyclic_avgpool5_backward      PhysicalDownsample, model/blocks.py:57-71

Each op has a fake (meta) implementation and an autograd formula, so it works under
``torch.compile(fullgraph=True)``, non-reentrant activation checkpointing (nothing but
the inputs is saved; the trajectory is recomputed in backward) and bf16 autocast.
CUDA only: there is no CPU implementation.

Forward-mode AD (``torch.func.jvp``, ``torch.autograd.forward_ad``) works through every public wrapper: when an input
carries a tangent, the wrapper calls its op through an autograd.Function with a jvp rule (sl_advect: the fused
tangent-linear kernel on the full mesh; the GeoCyclic ops: compositions of their own kernels).  Without a tangent the
op is called directly, as before.  vmap / jacfwd over a tangent, forward-over-reverse and tangents on latitude-band
geometries raise NotImplementedError.

Storage types of sl_advect.  The arithmetic is always fp32 (torch's own autocast policy runs
grid_sampler / asin / atan2 in fp32) and ``out`` is fp32.  When field, u and v are all bf16 (what
autocast hands the op: down_projection and velocity_net outputs) on the full mesh, with W % 8 == 0,
16-byte aligned bases and batch strides in multiples of 8 elements, the kernels read them as bf16 and
write bf16 gradients (``paradis::sl_advect_backward_bf16``, include/paradis_sl_bf16.h): no fp32 copy is
made, and the results are bit-identical to the fp32 op on ``.float()`` copies with the gradients cast
back by ``.to(torch.bfloat16)``.  Any other combination (fp16, mixed dtypes, latitude bands, other
alignments) is upcast to fp32 and the gradients are cast back to the input dtypes.

Storage types of geocyclic_pad, geocyclic_dwconv and geocyclic_avgpool5.  When the large tensors are bf16 (the input,
and grad_y in backward), the kernels read and write bf16 (include/paradis_geocyclic.h); weight and bias stay fp32 (a
bf16 weight of C * k * k elements is upcast) and so do grad weight / grad bias.  The results are bit-identical to the
fp32 kernels run on ``.float()`` copies with the outputs cast back by ``.to(torch.bfloat16)``.  fp16, fp32 and
mixed-dtype calls take the fp32 kernels (on fp32 copies where needed).  ``NATIVE_BF16 = False`` forces the upcast path
for these ops as well.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import List, Optional, Tuple

import torch
import torch.autograd.forward_ad as fwAD
from torch import Tensor
from torch._C._functorch import TransformType
from torch._functorch.pyfunctorch import retrieve_all_functorch_interpreters

from . import _lib

__all__ = ["SLGeometry", "sl_advect", "geocyclic_pad", "geocyclic_dwconv", "geocyclic_avgpool5", "check_status",
           "poll_status", "host_fwd_bwd"]

_status_words: dict = {}


def _status_word(device: torch.device) -> Tensor:
    """One int32 per device in MAPPED PINNED HOST memory (cudaHostAlloc memory is device-accessible
    under UVA): a kernel that detects a contract violation stores the code straight into host memory,
    so the host can look at it at the start of every later call without a synchronisation or a copy."""
    key = (device.type, device.index if device.index is not None else torch.cuda.current_device())
    if key not in _status_words:
        _status_words[key] = torch.zeros(1, dtype=torch.int32).pin_memory()
    return _status_words[key]


def _raise_status(word: Tensor) -> None:
    code = int(word[0])
    word.zero_()
    raise RuntimeError(f"paradis_sl device status {_lib.STATUS_NAMES.get(code, code)}: "
                       "semi-Lagrangian displacement outside the supported window (more than "
                       f"{_lib.MAX_DISP_ROWS} rows, or a departure stencil outside a latitude band's halo) "
                       "in this or an earlier call on this device")


def poll_status(device) -> None:
    """Non-blocking check, run at the start of every operator call: raises if a kernel of an EARLIER call has
    reported a contract violation by now.  Costs one host memory read."""
    word = _status_word(torch.device(device))
    if int(word[0]):
        _raise_status(word)


def check_status(device=None) -> None:
    """Synchronise and raise if a kernel flagged a device-side contract violation
    (displacement above 126 rows, or a departure stencil outside the rows held by
    ``field`` in a latitude-band call)."""
    device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    word = _status_word(device)
    torch.cuda.synchronize(device)
    if int(word[0]):
        _raise_status(word)


def _stream(t: Tensor) -> C.c_void_p:
    return C.c_void_p(torch.cuda.current_stream(t.device).cuda_stream)


def _ptr(t) -> C.c_void_p:
    return C.c_void_p(0 if t is None else t.data_ptr())


def _inner_contig(t: Tensor) -> Tensor:
    """Accept batch-strided views (model/paradis.py:235-237) without copying."""
    _, V, R, W = t.shape
    if t.stride(3) == 1 and t.stride(2) == W and t.stride(1) == R * W and t.stride(0) >= 0:
        return t
    return t.contiguous()


def _hpad(H: int) -> int:
    return (H + 3) // 4 * 4


def pack_tables(lat: Tensor, lon: Tensor) -> Tensor:
    """[sin(lat) | cos(lat) | lon], fp32, latitude sections zero-padded to 4-entry multiples.
    sin/cos run as torch fp32 kernels on the device of ``lat`` (what the reference evaluates
    on its ``lat_grid`` buffer, advection.py:86-87)."""
    H, Hp = lat.numel(), _hpad(lat.numel())
    t = torch.zeros(2 * Hp + lon.numel(), dtype=torch.float32, device=lat.device)
    t[:H] = torch.sin(lat.float())
    t[Hp:Hp + H] = torch.cos(lat.float())
    t[2 * Hp:] = lon.float()
    return t


class SLGeometry:
    """Separable mesh geometry: what model/advection.py:56-72 registers as buffers.

    ``tables`` = [sin(lat) | cos(lat) | lon] in fp32 on the compute device, the two latitude
    sections padded to a multiple of 4 entries so every section is 16-byte aligned,
    ``scalars`` = [min_lat, d_lat, min_lon, d_lon] (fp32 values as python floats),
    ``windows`` = [H, W, own0, ownN, arr0, arrN, fld0, fldN] (latitude-band decomposition;
    full mesh by default), optionally followed by [peer_lo_ptr, peer_hi_ptr, peer_rows]: device
    addresses of the latitude neighbours' boundary rows of `field` (NVLink peer memory, see
    include/paradis_sl.h) which the kernels then read in place instead of an assembled halo.
    """

    def __init__(self, tables: Tensor, scalars: List[float], H: int, W: int, windows=None):
        self.tables = tables
        self.scalars = [float(s) for s in scalars]
        self.H, self.W = int(H), int(W)
        self.windows = list(windows) if windows is not None else [self.H, self.W, 0, self.H, 0, self.H, 0, self.H]

    @staticmethod
    def separable(lat_grid: Tensor, lon_grid: Tensor) -> bool:
        return bool((lat_grid == lat_grid[:, :1]).all()) and bool((lon_grid == lon_grid[:1, :]).all())

    @classmethod
    def from_grids(cls, lat_grid: Tensor, lon_grid: Tensor) -> "SLGeometry":
        """lat_grid, lon_grid: [H, W] radians, as data/era5_dataset.py:178-182 builds them.
        sin/cos are taken with torch on the device the grids live on, i.e. the same fp32
        kernels the reference applies to its ``lat_grid`` buffer (advection.py:86-87)."""
        if lat_grid.dim() != 2 or lat_grid.shape != lon_grid.shape:
            raise ValueError("lat_grid and lon_grid must be [H, W]")
        if not cls.separable(lat_grid, lon_grid):
            raise ValueError("paradis_sl needs a separable lat-lon mesh (lat constant along W, lon along H)")
        H, W = lat_grid.shape
        lat = lat_grid[:, 0].to(torch.float32).contiguous()
        lon = lon_grid[0, :].to(torch.float32).contiguous()
        tables = pack_tables(lat, lon)
        lat_min, lat_max = lat.min(), lat.max()
        lon_min, lon_max = lon.min(), lon.max()
        scalars = [lat_min.item(), (lat_max - lat_min).item(), lon_min.item(), (lon_max - lon_min).item()]
        return cls(tables, scalars, H, W)

    def to(self, device) -> "SLGeometry":
        return SLGeometry(self.tables.to(device), self.scalars, self.H, self.W, self.windows)

    def band(self, own: Tuple[int, int], arr: Tuple[int, int], fld: Tuple[int, int], peer=None,
             arr_peer=None) -> "SLGeometry":
        """Same mesh, different row windows (row0, rows) for a latitude band; ``peer`` =
        (lo_ptr, hi_ptr, rows) for field halos read in place from the neighbours; ``arr_peer`` =
        ([lo_u, lo_v, lo_g], [hi_u, hi_v, hi_g], rows) likewise for u, v, grad_out in the backward."""
        w = [self.H, self.W, own[0], own[1], arr[0], arr[1], fld[0], fld[1]]
        if peer is not None or arr_peer is not None:
            w += [int(peer[0]), int(peer[1]), int(peer[2])] if peer is not None else [0, 0, 0]
        if arr_peer is not None:
            w += [int(p) for p in arr_peer[0]] + [int(p) for p in arr_peer[1]] + [int(arr_peer[2])]
        return SLGeometry(self.tables, self.scalars, self.H, self.W, w)


def _geom_struct(tables: Tensor, scalars: List[float], windows: List[int]) -> _lib.Geom:
    H, W = int(windows[0]), int(windows[1])
    Hp = _hpad(H)
    if tables.dtype != torch.float32 or tables.numel() != 2 * Hp + W or not tables.is_contiguous():
        raise RuntimeError("paradis_sl: geometry tables must be a contiguous fp32 tensor from pack_tables()")
    base = tables.data_ptr()
    g = _lib.Geom()
    g.H, g.W = H, W
    g.sin_lat, g.cos_lat, g.lon = base, base + 4 * Hp, base + 8 * Hp
    g.min_lat, g.d_lat, g.min_lon, g.d_lon = scalars
    g.own_row0, g.own_rows, g.arr_row0, g.arr_rows, g.fld_row0, g.fld_rows = [int(w) for w in windows[2:8]]
    if len(windows) >= 11:
        g.fld_peer_lo, g.fld_peer_hi, g.fld_peer_rows = (int(windows[8]) or None), (int(windows[9]) or None), int(windows[10])
    if len(windows) >= 18:
        for k in range(3):
            g.arr_peer_lo[k] = int(windows[11 + k]) or None
            g.arr_peer_hi[k] = int(windows[14 + k]) or None
        g.arr_peer_rows = int(windows[17])
    return g


def _held_arr_rows(windows: List[int]) -> int:
    """Rows the u / v / grad_out tensors hold: the arr window minus the peer halos (if any)."""
    n = int(windows[5])
    if len(windows) >= 18 and int(windows[17]) > 0:
        h = int(windows[17])
        n -= (h if int(windows[11]) else 0) + (h if int(windows[14]) else 0)
    return n


def _check_inputs(field: Tensor, u: Tensor, v: Tensor, windows: List[int]):
    if not (field.is_cuda and u.is_cuda and v.is_cuda):
        raise RuntimeError("paradis::sl_advect is a CUDA-only operator (no CPU fallback)")
    if field.dim() != 4 or u.shape != v.shape or u.dim() != 4:
        raise RuntimeError("paradis::sl_advect expects field [B,V,Rf,W] and u, v [B,V,Ra,W]")
    H, W, own0, ownN, arr0, arrN, fld0, fldN = [int(w) for w in windows[:8]]
    B, V = field.shape[:2]
    if tuple(field.shape) != (B, V, fldN, W) or tuple(u.shape) != (B, V, _held_arr_rows(windows), W):
        raise RuntimeError(f"paradis::sl_advect shape mismatch: field {tuple(field.shape)}, u {tuple(u.shape)}, "
                           f"windows {windows}")
    return B, V, H, W, ownN, arrN


def _full_mesh(windows: List[int]) -> bool:
    H = int(windows[0])
    return len(windows) == 8 and [int(w) for w in windows[2:8]] == [0, H, 0, H, 0, H]


def _bf16_candidate(dtypes, windows: List[int]) -> bool:
    """What the native bf16 path needs that is known without the data (dtypes, windows, W): safe in traced code."""
    return (NATIVE_BF16 and all(d == torch.bfloat16 for d in dtypes) and _full_mesh(windows)
            and int(windows[1]) % 8 == 0)


def _geo_bf16(*tensors: Tensor) -> bool:
    """Native bf16 storage of the GeoCyclic ops: every large tensor is bf16.  Decided from dtypes only (call time, safe
    in traced code)."""
    return NATIVE_BF16 and all(t.dtype == torch.bfloat16 for t in tensors)


def _bf16_layout_ok(bf: List[Tensor], f32: List[Tensor]) -> bool:
    """Alignment part of the native bf16 rule: 16-byte bases, batch strides in multiples of 8 (bf16) / 4 (fp32)
    elements, so that every row starts on 16 bytes (include/paradis_sl_bf16.h)."""
    return (all(t.data_ptr() % 16 == 0 and t.stride(0) % 8 == 0 for t in bf)
            and all(t.data_ptr() % 16 == 0 and t.stride(0) % 4 == 0 for t in f32))


# --------------------------------------------------------------------------------------
# forward-mode AD.  torch gives a custom op no forward-AD formula (its tangent would come out None or zero), so a
# public wrapper whose inputs carry a tangent (torch.autograd.forward_ad or torch.func.jvp) calls the op through an
# autograd.Function with a jvp rule instead.  Calls without a tangent call the op directly: dynamo refuses an
# autograd.Function that defines jvp, and compiled training steps must not break their graph.
# --------------------------------------------------------------------------------------
def _has_tangent(*tensors) -> bool:
    return any(t is not None and fwAD.unpack_dual(t).tangent is not None for t in tensors)


def _transforms() -> list:
    """The functorch transforms active around this call (outermost first); none while dynamo traces."""
    if torch.compiler.is_compiling():
        return []
    return [i.key() for i in retrieve_all_functorch_interpreters()]


def _tangent_path(*tensors) -> bool:
    """True when an input carries a forward-mode tangent: the call must take the autograd.Function with a jvp rule.
    Raises NotImplementedError where no rule exists (vmap / jacfwd, forward-over-reverse)."""
    if _has_tangent(*tensors):
        if TransformType.Vmap in _transforms():
            raise NotImplementedError("paradis ops have no vmap rule: torch.func.vmap / jacfwd over a forward-mode tangent "
                                      "is not supported (use torch.func.jvp or torch.autograd.forward_ad per direction)")
        return True
    t = _transforms()
    if TransformType.Jvp in t and TransformType.Grad in t[t.index(TransformType.Jvp):]:
        raise NotImplementedError("paradis ops support forward mode (jvp) and reverse mode (vjp / grad), not forward-over-"
                                  "reverse: the backward ops have no tangent rule")
    return False


def _no_fwd_over_rev(*tensors) -> None:
    """Guard of the backward formulas: the backward ops have no tangent rule, so a tangent on grad_out or on a saved
    input (forward-over-reverse, e.g. Hessian-vector products) must not be dropped silently."""
    if _has_tangent(*tensors):
        raise NotImplementedError("paradis ops support forward mode (jvp) and reverse mode (vjp / grad), not forward-over-"
                                  "reverse: the backward ops have no tangent rule")


def _no_vmap(info, in_dims, *args):
    raise NotImplementedError("paradis ops have no vmap rule: torch.func.vmap / jacfwd over a forward-mode tangent is "
                              "not supported (use torch.func.jvp or torch.autograd.forward_ad per direction)")


# --------------------------------------------------------------------------------------
# sl_advect
# --------------------------------------------------------------------------------------
@torch.library.custom_op("paradis::sl_advect", mutates_args=(), device_types="cuda")
def _sl_advect(field: Tensor, u: Tensor, v: Tensor, tables: Tensor, scalars: List[float], dt: float,
               interp: int, pole_fix: bool, math: int, windows: List[int], cfl: float) -> Tensor:
    B, V, H, W, ownN, arrN = _check_inputs(field, u, v, windows)
    L = _lib.lib()
    if field.dtype == torch.float64 or u.dtype == torch.float64 or v.dtype == torch.float64:
        raise RuntimeError("paradis::sl_advect computes in fp32 (like the reference under its fp32 / bf16-mixed settings); "
                           "float64 inputs would silently lose precision -- cast them explicitly")
    poll_status(field.device)
    if tables.device != field.device:
        raise RuntimeError(f"paradis::sl_advect: geometry tables live on {tables.device}, the tensors on {field.device}; "
                           "move the geometry with SLGeometry.to(device)")
    native = _bf16_candidate((field.dtype, u.dtype, v.dtype), windows)
    if native:
        field, u, v = _inner_contig(field), _inner_contig(u), _inner_contig(v)
        native = _bf16_layout_ok([field, u, v], [])
    if not native:
        field = _inner_contig(field.float())
        u = _inner_contig(u.float())
        v = _inner_contig(v.float())
    out = torch.empty((B, V, ownN, W), dtype=torch.float32, device=field.device)
    g = _geom_struct(tables, scalars, windows)
    ws_bytes = L.paradis_sl_advect_fwd_workspace(B, V)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=field.device)
    fwd = L.paradis_sl_advect_fwd_bf16 if native else L.paradis_sl_advect_fwd
    with torch.cuda.device(field.device):
        rc = fwd(C.byref(g), _ptr(field), _ptr(u), _ptr(v), _ptr(out), B, V,
                 field.stride(0), u.stride(0), v.stride(0), dt, interp, int(pole_fix), math,
                 _ptr(ws), ws_bytes, _ptr(_status_word(field.device)), _stream(field))
    _lib.check(rc, "paradis_sl_advect_fwd_bf16" if native else "paradis_sl_advect_fwd")
    return out


@_sl_advect.register_fake
def _(field, u, v, tables, scalars, dt, interp, pole_fix, math, windows, cfl):
    B, V = field.shape[:2]
    return field.new_empty((B, V, windows[3], windows[1]), dtype=torch.float32)


def _backward_impl(grad_out: Tensor, field: Tensor, u: Tensor, v: Tensor, tables: Tensor, scalars: List[float],
                   dt: float, interp: int, pole_fix: bool, math: int, windows: List[int], cfl: float,
                   need_field: bool, need_uv: bool, native: bool, what: str):
    """Both backward ops.  native: bf16 field / u / v read in place, bf16 gradients (paradis_sl_advect_bwd_bf16);
    otherwise the inputs are upcast and the gradients are fp32.  Returns (gf, gu, gv, dtype of the gradients)."""
    B, V, H, W, ownN, arrN = _check_inputs(field, u, v, windows)
    L = _lib.lib()
    dev = field.device
    poll_status(dev)
    if tables.device != dev:
        raise RuntimeError(f"{what}: geometry tables live on {tables.device}, the tensors on {dev}")
    grad_out = _inner_contig(grad_out.float())
    if native:
        field, u, v = _inner_contig(field), _inner_contig(u), _inner_contig(v)
        native = _bf16_layout_ok([field, u, v], [grad_out])
    if not native:
        field = _inner_contig(field.float())
        u = _inner_contig(u.float())
        v = _inner_contig(v.float())
    if tuple(grad_out.shape) != tuple(u.shape):
        raise RuntimeError(f"{what}: grad_out must cover the arrival window like u and v")
    gdt = torch.bfloat16 if native else torch.float32
    gf = torch.empty((B, V, ownN, W), dtype=gdt, device=dev) if need_field else None
    gu = torch.empty((B, V, ownN, W), dtype=gdt, device=dev) if need_uv else None
    gv = torch.empty((B, V, ownN, W), dtype=gdt, device=dev) if need_uv else None
    g = _geom_struct(tables, scalars, windows)
    ws_bytes = (L.paradis_sl_advect_bwd_bf16_workspace if native else L.paradis_sl_advect_bwd_workspace)(B, V, arrN, W)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    bwd = L.paradis_sl_advect_bwd_bf16 if native else L.paradis_sl_advect_bwd
    with torch.cuda.device(dev):
        rc = bwd(C.byref(g), _ptr(grad_out), _ptr(field), _ptr(u), _ptr(v), _ptr(gf), _ptr(gu),
                 _ptr(gv), B, V, grad_out.stride(0), field.stride(0), u.stride(0), v.stride(0),
                 dt, interp, int(pole_fix), math, 3 | (8 if FORCE_ROW_SWEEP else 0), cfl, _ptr(ws),
                 ws_bytes, _ptr(_status_word(dev)), _stream(field))
    _lib.check(rc, "paradis_sl_advect_bwd_bf16" if native else "paradis_sl_advect_bwd")
    return gf, gu, gv, gdt


@torch.library.custom_op("paradis::sl_advect_backward", mutates_args=(), device_types="cuda")
def _sl_advect_backward(grad_out: Tensor, field: Tensor, u: Tensor, v: Tensor, tables: Tensor,
                        scalars: List[float], dt: float, interp: int, pole_fix: bool, math: int,
                        windows: List[int], cfl: float, need_field: bool,
                        need_uv: bool) -> Tuple[Tensor, Tensor, Tensor]:
    gf, gu, gv, _ = _backward_impl(grad_out, field, u, v, tables, scalars, dt, interp, pole_fix, math, windows, cfl,
                                   need_field, need_uv, False, "paradis::sl_advect_backward")
    none = lambda: torch.empty(0, dtype=torch.float32, device=field.device)
    return (gf if need_field else none(), gu if need_uv else none(), gv if need_uv else none())


@_sl_advect_backward.register_fake
def _(grad_out, field, u, v, tables, scalars, dt, interp, pole_fix, math, windows, cfl, need_field, need_uv):
    B, V = field.shape[:2]
    shape = (B, V, windows[3], windows[1])
    full = lambda: field.new_empty(shape, dtype=torch.float32)
    none = lambda: field.new_empty((0,), dtype=torch.float32)
    return (full() if need_field else none(), full() if need_uv else none(), full() if need_uv else none())


@torch.library.custom_op("paradis::sl_advect_backward_bf16", mutates_args=(), device_types="cuda")
def _sl_advect_backward_bf16(grad_out: Tensor, field: Tensor, u: Tensor, v: Tensor, tables: Tensor,
                             scalars: List[float], dt: float, interp: int, pole_fix: bool, math: int,
                             windows: List[int], cfl: float, need_field: bool,
                             need_uv: bool) -> Tuple[Tensor, Tensor, Tensor]:
    """Backward of sl_advect for bf16 field / u / v: bf16 gradients.  Read in place by the bf16 kernels when the
    layout allows it (see the module docstring), otherwise computed from fp32 copies and rounded by .to()."""
    native = _bf16_candidate((field.dtype, u.dtype, v.dtype), windows)
    gf, gu, gv, gdt = _backward_impl(grad_out, field, u, v, tables, scalars, dt, interp, pole_fix, math, windows, cfl,
                                     need_field, need_uv, native, "paradis::sl_advect_backward_bf16")
    if gdt != torch.bfloat16:
        gf, gu, gv = [t.to(torch.bfloat16) if t is not None else None for t in (gf, gu, gv)]
    none = lambda: torch.empty(0, dtype=torch.bfloat16, device=field.device)
    return (gf if need_field else none(), gu if need_uv else none(), gv if need_uv else none())


@_sl_advect_backward_bf16.register_fake
def _(grad_out, field, u, v, tables, scalars, dt, interp, pole_fix, math, windows, cfl, need_field, need_uv):
    B, V = field.shape[:2]
    shape = (B, V, windows[3], windows[1])
    full = lambda: field.new_empty(shape, dtype=torch.bfloat16)
    none = lambda: field.new_empty((0,), dtype=torch.bfloat16)
    return (full() if need_field else none(), full() if need_uv else none(), full() if need_uv else none())


def _sl_setup(ctx, inputs, output):
    field, u, v, tables, scalars, dt, interp, pole_fix, math, windows, cfl = inputs
    ctx.save_for_backward(field, u, v, tables)
    ctx.attrs = (scalars, dt, interp, pole_fix, math, windows, cfl)
    ctx.dtypes = (field.dtype, u.dtype, v.dtype)


def _sl_backward(ctx, grad_out):
    field, u, v, tables = ctx.saved_tensors
    _no_fwd_over_rev(grad_out, field, u, v)
    scalars, dt, interp, pole_fix, math, windows, cfl = ctx.attrs
    if list(windows[2:4]) != list(windows[4:6]):
        raise RuntimeError("autograd through a latitude-band sl_advect needs halo'd grad_out: "
                           "use paradis_model_b200.halo.LatBandAdvection")
    need_field = ctx.needs_input_grad[0]
    need_uv = ctx.needs_input_grad[1] or ctx.needs_input_grad[2]
    # bf16 inputs on the full mesh: bf16 gradients straight from the kernels (no fp32 copies, no casts)
    bwd = (torch.ops.paradis.sl_advect_backward_bf16 if _bf16_candidate(ctx.dtypes, windows)
           else torch.ops.paradis.sl_advect_backward)
    gf, gu, gv = bwd(grad_out, field, u, v, tables, scalars, dt, interp, pole_fix, math, windows, cfl, need_field,
                     need_uv)
    gf = gf.to(ctx.dtypes[0]) if need_field else None
    gu = gu.to(ctx.dtypes[1]) if ctx.needs_input_grad[1] else None
    gv = gv.to(ctx.dtypes[2]) if ctx.needs_input_grad[2] else None
    return gf, gu, gv, None, None, None, None, None, None, None, None


_sl_advect.register_autograd(_sl_backward, setup_context=_sl_setup)


@torch.library.custom_op("paradis::sl_advect_jvp", mutates_args=(), device_types="cuda")
def _sl_advect_jvp(field: Tensor, u: Tensor, v: Tensor, dfield: Optional[Tensor], du: Tensor, dv: Tensor,
                   tables: Tensor, scalars: List[float], dt: float, interp: int, pole_fix: bool, math: int,
                   windows: List[int]) -> Tensor:
    """Tangent-linear model of sl_advect (include/paradis_sl_tl.h): d out along (dfield, du, dv), fp32.  dfield may be
    None (velocity tangents only).  Full mesh only; every input is read as fp32 (bf16 / fp16 are upcast)."""
    B, V, H, W, ownN, arrN = _check_inputs(field, u, v, windows)
    if not _full_mesh(windows):
        raise RuntimeError("paradis::sl_advect_jvp works on the full mesh only")
    for name, t in (("dfield", dfield), ("du", du), ("dv", dv)):
        if t is not None and tuple(t.shape) != tuple(field.shape if name == "dfield" else u.shape):
            raise RuntimeError(f"paradis::sl_advect_jvp: {name} {tuple(t.shape)} does not match its primal")
    if any(t is not None and t.dtype == torch.float64 for t in (field, u, v, dfield, du, dv)):
        raise RuntimeError("paradis::sl_advect_jvp computes in fp32; cast float64 inputs explicitly")
    poll_status(field.device)
    if tables.device != field.device:
        raise RuntimeError(f"paradis::sl_advect_jvp: geometry tables live on {tables.device}, the tensors on {field.device}")
    field, u, v, du, dv = [_inner_contig(t.float()) for t in (field, u, v, du, dv)]
    dfield = _inner_contig(dfield.float()) if dfield is not None else None
    L = _lib.lib()
    dout = torch.empty((B, V, ownN, W), dtype=torch.float32, device=field.device)
    g = _geom_struct(tables, scalars, windows)
    ws_bytes = L.paradis_sl_advect_jvp_workspace(B, V)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=field.device)
    with torch.cuda.device(field.device):
        rc = L.paradis_sl_advect_jvp(C.byref(g), _ptr(field), _ptr(dfield), _ptr(u), _ptr(v), _ptr(du), _ptr(dv),
                                     _ptr(dout), B, V, field.stride(0), dfield.stride(0) if dfield is not None else 0,
                                     u.stride(0), v.stride(0), du.stride(0), dv.stride(0), dt, interp, int(pole_fix),
                                     math, _ptr(ws), ws_bytes, _ptr(_status_word(field.device)), _stream(field))
    _lib.check(rc, "paradis_sl_advect_jvp")
    return dout


@_sl_advect_jvp.register_fake
def _(field, u, v, dfield, du, dv, tables, scalars, dt, interp, pole_fix, math, windows):
    B, V = field.shape[:2]
    return field.new_empty((B, V, windows[3], windows[1]), dtype=torch.float32)


class _SLAdvectFn(torch.autograd.Function):
    """paradis::sl_advect with a jvp rule (forward-mode AD); same setup and backward as the op's own autograd."""

    @staticmethod
    def forward(field, u, v, tables, scalars, dt, interp, pole_fix, math, windows, cfl):
        return torch.ops.paradis.sl_advect(field, u, v, tables, scalars, dt, interp, pole_fix, math, windows, cfl)

    @staticmethod
    def setup_context(ctx, inputs, output):
        _sl_setup(ctx, inputs, output)
        ctx.save_for_forward(*inputs[:4])
        ctx.set_materialize_grads(False)        # inputs without a tangent reach jvp as None, not as zeros

    backward = staticmethod(_sl_backward)
    vmap = staticmethod(_no_vmap)

    @staticmethod
    def jvp(ctx, dfield, du, dv, *_):
        field, u, v, tables = ctx.saved_tensors
        scalars, dt, interp, pole_fix, math, windows, cfl = ctx.attrs
        if du is None and dv is None:        # the op is linear in field: its tangent is the op applied to dfield
            return torch.ops.paradis.sl_advect(dfield, u, v, tables, scalars, dt, interp, pole_fix, math, windows, cfl)
        du = du if du is not None else torch.zeros_like(u)
        dv = dv if dv is not None else torch.zeros_like(v)
        return torch.ops.paradis.sl_advect_jvp(field, u, v, dfield, du, dv, tables, scalars, dt, interp, pole_fix,
                                               math, windows)


DEFAULT_CFL_CELLS = 8.0
FORCE_ROW_SWEEP = False     # tests: run the row-sweep backward also where the strip sweep is the default (PARADIS_BWD_ROWSWEEP)
NATIVE_BF16 = True          # bf16 field / u / v read and bf16 gradients written by the kernels where eligible, and bf16
                            # storage in the geocyclic pad / dwconv / avgpool5 kernels (read at call time; False runs
                            # the upcast path, for tests and timings of the two in one process)
# read once at import (not inside traced code): PARADIS_SL_MATH=fast|exact overrides the math mode,
# PARADIS_SL_CHECK=1 synchronises after every call and raises on a device-side contract violation
_ENV_MATH = os.environ.get("PARADIS_SL_MATH", "")
_ENV_CHECK = os.environ.get("PARADIS_SL_CHECK") == "1"


def sl_advect(field: Tensor, u: Tensor, v: Tensor, geometry: SLGeometry, dt: float,
              interpolation: str = "bilinear", pole_fix: bool = True, math: str = "fast",
              cfl_cells: float = DEFAULT_CFL_CELLS) -> Tensor:
    """Fused operator core: drop-in for model/advection.py:129-169.

    field, u, v : [B, V, H, W] CUDA tensors (u, v may be batch-strided views).  Differentiable
    w.r.t. all three; the backward is deterministic.  ``math="exact"`` replays the reference's
    fp32 operation order for the departure coordinates.  ``cfl_cells`` is a performance hint
    for the backward (expected bound on |(u, v)| * dt in latitude cells): planes that exceed it
    are detected on the device and recomputed by the general path, results never depend on it;
    ``0`` disables the fused backward.

    Forward-mode AD (``torch.func.jvp``, ``torch.autograd.forward_ad``) gives the tangent-linear model on the full
    mesh, in fp32 (``paradis::sl_advect_jvp``).
    """
    if _ENV_MATH:
        math = _ENV_MATH
    args = (geometry.tables, geometry.scalars, float(dt), _lib.INTERP[interpolation], bool(pole_fix), _lib.MATH[math],
            geometry.windows, float(cfl_cells))
    if _tangent_path(field, u, v):
        if not _full_mesh(geometry.windows):
            raise NotImplementedError("forward-mode AD through sl_advect is supported on the full mesh only, not on "
                                      "latitude-band geometries")
        out = _SLAdvectFn.apply(field, u, v, *args)
    else:
        out = torch.ops.paradis.sl_advect(field, u, v, *args)
    if _ENV_CHECK:
        check_status(field.device)
    return out


# --------------------------------------------------------------------------------------
# geocyclic_pad
# --------------------------------------------------------------------------------------
@torch.library.custom_op("paradis::geocyclic_pad", mutates_args=(), device_types="cuda")
def _geocyclic_pad(x: Tensor, p: int) -> Tensor:
    if not x.is_cuda:
        raise RuntimeError("paradis::geocyclic_pad is a CUDA-only operator (no CPU fallback)")
    B, Cn, H, W = x.shape
    native = _geo_bf16(x)
    xs = x.contiguous() if native else x.float().contiguous()
    y = torch.empty((B, Cn, H + 2 * p, W + 2 * p), dtype=xs.dtype, device=x.device)
    name = "paradis_geocyclic_pad_fwd_bf16" if native else "paradis_geocyclic_pad_fwd"
    with torch.cuda.device(x.device):
        rc = getattr(_lib.lib(), name)(_ptr(xs), _ptr(y), B * Cn, H, W, p, _stream(x))
    _lib.check(rc, name)
    return y.to(x.dtype)


@_geocyclic_pad.register_fake
def _(x, p):
    B, Cn, H, W = x.shape
    return x.new_empty((B, Cn, H + 2 * p, W + 2 * p))


@torch.library.custom_op("paradis::geocyclic_pad_backward", mutates_args=(), device_types="cuda")
def _geocyclic_pad_backward(gy: Tensor, p: int) -> Tensor:
    B, Cn, Hp, Wp = gy.shape
    H, W = Hp - 2 * p, Wp - 2 * p
    native = _geo_bf16(gy)
    gs = gy.contiguous() if native else gy.float().contiguous()
    gx = torch.empty((B, Cn, H, W), dtype=gs.dtype, device=gy.device)
    name = "paradis_geocyclic_pad_bwd_bf16" if native else "paradis_geocyclic_pad_bwd"
    with torch.cuda.device(gy.device):
        rc = getattr(_lib.lib(), name)(_ptr(gs), _ptr(gx), B * Cn, H, W, p, _stream(gy))
    _lib.check(rc, name)
    return gx.to(gy.dtype)


@_geocyclic_pad_backward.register_fake
def _(gy, p):
    B, Cn, Hp, Wp = gy.shape
    return gy.new_empty((B, Cn, Hp - 2 * p, Wp - 2 * p))


def _pad_setup(ctx, inputs, output):
    ctx.p = inputs[1]


def _pad_backward(ctx, gy):
    _no_fwd_over_rev(gy)
    return torch.ops.paradis.geocyclic_pad_backward(gy, ctx.p), None


_geocyclic_pad.register_autograd(_pad_backward, setup_context=_pad_setup)


class _PadFn(torch.autograd.Function):
    """paradis::geocyclic_pad with a jvp rule: the op is linear, its tangent is the op applied to the tangent."""

    @staticmethod
    def forward(x, p):
        return torch.ops.paradis.geocyclic_pad(x, p)

    setup_context = staticmethod(_pad_setup)
    backward = staticmethod(_pad_backward)
    vmap = staticmethod(_no_vmap)

    @staticmethod
    def jvp(ctx, dx, _):
        return torch.ops.paradis.geocyclic_pad(dx, ctx.p)


def geocyclic_pad(x: Tensor, pad_width: int) -> Tensor:
    """model/padding.py:11-39 as one kernel (identity when pad_width == 0)."""
    if pad_width == 0:
        return x
    assert x.dim() == 4, "Input must be 4-dimensional [batch, channels, lat, lon]"
    assert x.shape[3] % 2 == 0, "Number of longitude points must be even"
    if _tangent_path(x):
        return _PadFn.apply(x, int(pad_width))
    return torch.ops.paradis.geocyclic_pad(x, int(pad_width))


# --------------------------------------------------------------------------------------
# geocyclic_dwconv: GeoCyclic padding fused into the depthwise convolution of SepConv (blocks.py:92-116)
# --------------------------------------------------------------------------------------
@torch.library.custom_op("paradis::geocyclic_dwconv", mutates_args=(), device_types="cuda")
def _geocyclic_dwconv(x: Tensor, weight: Tensor, bias: Optional[Tensor]) -> Tensor:
    B, Cn, H, W = x.shape
    k = weight.shape[-1]
    if tuple(weight.shape) != (Cn, 1, k, k):
        raise RuntimeError("paradis::geocyclic_dwconv expects a depthwise weight [C, 1, k, k]")
    native = _geo_bf16(x)
    xs = x.contiguous() if native else x.float().contiguous()
    wf = weight.float().contiguous()
    bf = bias.float().contiguous() if bias is not None else None
    y = torch.empty_like(xs)
    name = "paradis_geocyclic_dwconv_fwd_bf16" if native else "paradis_geocyclic_dwconv_fwd"
    with torch.cuda.device(x.device):
        rc = getattr(_lib.lib(), name)(_ptr(xs), _ptr(wf), _ptr(bf), _ptr(y), B, Cn, H, W, k, _stream(x))
    _lib.check(rc, name)
    return y.to(x.dtype)


@_geocyclic_dwconv.register_fake
def _(x, weight, bias):
    return torch.empty_like(x)


def _dw_backward_impl(gy: Tensor, x: Tensor, weight: Tensor, need_input: bool, need_weight: bool, need_bias: bool,
                      native: bool):
    """Both backward ops.  native: bf16 gy / x read in place and a bf16 grad input; otherwise fp32 copies and an fp32
    grad input.  grad weight / grad bias are fp32 either way.  Only the requested gradients are computed (a constant
    filter skips the weight-gradient pass and its workspace)."""
    B, Cn, H, W = x.shape
    k = weight.shape[-1]
    L = _lib.lib()
    gs = gy.contiguous() if native else gy.float().contiguous()
    wf = weight.float().contiguous()
    sfx = "_bf16" if native else ""
    empty = lambda: torch.empty(0, dtype=torch.float32, device=x.device)
    gx, gw, gb = empty(), empty(), empty()
    with torch.cuda.device(x.device):
        if need_input:
            gx = torch.empty((B, Cn, H, W), dtype=gs.dtype, device=x.device)
            name = "paradis_geocyclic_dwconv_bwd_input" + sfx
            rc = getattr(L, name)(_ptr(gs), _ptr(wf), _ptr(gx), B, Cn, H, W, k, _stream(x))
            _lib.check(rc, name)
        if need_weight or need_bias:
            xs = x.contiguous() if native else x.float().contiguous()
            gw = torch.empty_like(wf)
            gb = torch.empty(Cn if need_bias else 0, dtype=torch.float32, device=x.device)
            ws_bytes = L.paradis_geocyclic_dwconv_wgrad_workspace(B, Cn, H, W, k)
            ws = torch.empty(ws_bytes, dtype=torch.uint8, device=x.device)
            name = "paradis_geocyclic_dwconv_bwd_weight" + sfx
            rc = getattr(L, name)(_ptr(xs), _ptr(gs), _ptr(gw), _ptr(gb) if need_bias else _ptr(None),
                                  B, Cn, H, W, k, _ptr(ws), ws_bytes, _stream(x))
            _lib.check(rc, name)
    return gx, gw, gb


@torch.library.custom_op("paradis::geocyclic_dwconv_backward", mutates_args=(), device_types="cuda")
def _geocyclic_dwconv_backward(gy: Tensor, x: Tensor, weight: Tensor, need_input: bool, need_weight: bool,
                               need_bias: bool) -> Tuple[Tensor, Tensor, Tensor]:
    """fp32 gradients from fp32 copies of gy and x."""
    return _dw_backward_impl(gy, x, weight, need_input, need_weight, need_bias, False)


@_geocyclic_dwconv_backward.register_fake
def _(gy, x, weight, need_input, need_weight, need_bias):
    none = lambda: x.new_empty((0,), dtype=torch.float32)
    return (torch.empty_like(x, dtype=torch.float32) if need_input else none(),
            torch.empty_like(weight, dtype=torch.float32) if (need_weight or need_bias) else none(),
            x.new_empty((x.shape[1],), dtype=torch.float32) if need_bias else none())


@torch.library.custom_op("paradis::geocyclic_dwconv_backward_bf16", mutates_args=(), device_types="cuda")
def _geocyclic_dwconv_backward_bf16(gy: Tensor, x: Tensor, weight: Tensor, need_input: bool, need_weight: bool,
                                    need_bias: bool) -> Tuple[Tensor, Tensor, Tensor]:
    """Backward for a bf16 x: bf16 grad input, fp32 grad weight / grad bias.  gy and x are read in place by the bf16
    kernels when both are bf16, otherwise the grad input is computed from fp32 copies and rounded by .to()."""
    native = _geo_bf16(gy, x)
    gx, gw, gb = _dw_backward_impl(gy, x, weight, need_input, need_weight, need_bias, native)
    gx = gx.to(torch.bfloat16) if need_input else torch.empty(0, dtype=torch.bfloat16, device=x.device)
    return gx, gw, gb


@_geocyclic_dwconv_backward_bf16.register_fake
def _(gy, x, weight, need_input, need_weight, need_bias):
    none = lambda dt: x.new_empty((0,), dtype=dt)
    return (torch.empty_like(x, dtype=torch.bfloat16) if need_input else none(torch.bfloat16),
            torch.empty_like(weight, dtype=torch.float32) if (need_weight or need_bias) else none(torch.float32),
            x.new_empty((x.shape[1],), dtype=torch.float32) if need_bias else none(torch.float32))


def _dw_setup(ctx, inputs, output):
    x, weight, bias = inputs
    ctx.save_for_backward(x, weight)
    ctx.has_bias = bias is not None
    ctx.dtypes = (x.dtype, weight.dtype, bias.dtype if bias is not None else None)


def _dw_backward(ctx, gy):
    x, weight = ctx.saved_tensors
    _no_fwd_over_rev(gy, x, weight)
    need_x, need_w = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
    need_b = ctx.has_bias and ctx.needs_input_grad[2]
    if not (need_x or need_w or need_b):
        return None, None, None
    # bf16 x and grad_y: bf16 grad input straight from the kernels (no fp32 copies, no casts)
    bwd = (torch.ops.paradis.geocyclic_dwconv_backward_bf16 if _geo_bf16(gy) and ctx.dtypes[0] == torch.bfloat16
           else torch.ops.paradis.geocyclic_dwconv_backward)
    gx, gw, gb = bwd(gy, x, weight, need_x, need_w, need_b)
    return (gx.to(ctx.dtypes[0]) if need_x else None, gw.to(ctx.dtypes[1]) if need_w else None,
            gb.to(ctx.dtypes[2]) if need_b else None)


_geocyclic_dwconv.register_autograd(_dw_backward, setup_context=_dw_setup)


class _DwConvFn(torch.autograd.Function):
    """paradis::geocyclic_dwconv with a jvp rule.  The op is bilinear in (x, weight) and affine in bias:
    d y = dwconv(dx, w) + dwconv(x, dw) + db, each term summed in fp32 and rounded once to y's dtype."""

    @staticmethod
    def forward(x, weight, bias):
        return torch.ops.paradis.geocyclic_dwconv(x, weight, bias)

    @staticmethod
    def setup_context(ctx, inputs, output):
        _dw_setup(ctx, inputs, output)
        ctx.save_for_forward(inputs[0], inputs[1])
        ctx.set_materialize_grads(False)        # inputs without a tangent reach jvp as None, not as zeros

    backward = staticmethod(_dw_backward)
    vmap = staticmethod(_no_vmap)

    @staticmethod
    def jvp(ctx, dx, dw, db):
        x, weight = ctx.saved_tensors
        terms = []
        if dx is not None:
            terms.append(torch.ops.paradis.geocyclic_dwconv(dx, weight, None).float())
        if dw is not None:
            terms.append(torch.ops.paradis.geocyclic_dwconv(x, dw, None).float())
        if db is not None and ctx.has_bias:
            terms.append(db.float().view(1, -1, 1, 1).expand(x.shape))
        dy = terms[0]
        for t in terms[1:]:
            dy = dy + t
        return dy.to(x.dtype).contiguous()


# --------------------------------------------------------------------------------------
# geocyclic_avgpool5: PhysicalDownsample (blocks.py:57-71), strided outputs only
# --------------------------------------------------------------------------------------
@torch.library.custom_op("paradis::geocyclic_avgpool5", mutates_args=(), device_types="cuda")
def _geocyclic_avgpool5(x: Tensor, stride: int) -> Tensor:
    B, Cn, H, W = x.shape
    native = _geo_bf16(x)
    xs = x.contiguous() if native else x.float().contiguous()
    y = torch.empty((B, Cn, (H - 1) // stride + 1, (W - 1) // stride + 1), dtype=xs.dtype, device=x.device)
    name = "paradis_geocyclic_avgpool5_fwd_bf16" if native else "paradis_geocyclic_avgpool5_fwd"
    with torch.cuda.device(x.device):
        rc = getattr(_lib.lib(), name)(_ptr(xs), _ptr(y), B, Cn, H, W, stride, _stream(x))
    _lib.check(rc, name)
    return y.to(x.dtype)


@_geocyclic_avgpool5.register_fake
def _(x, stride):
    B, Cn, H, W = x.shape
    return x.new_empty((B, Cn, (H - 1) // stride + 1, (W - 1) // stride + 1))


@torch.library.custom_op("paradis::geocyclic_avgpool5_backward", mutates_args=(), device_types="cuda")
def _geocyclic_avgpool5_backward(gy: Tensor, H: int, W: int, stride: int) -> Tensor:
    """Adjoint of geocyclic_avgpool5 for an [B, C, H, W] input: one kernel that gathers, for every input point, the
    strided outputs whose 5x5 window covers it.  Returns gy's dtype."""
    B, Cn, Ho, Wo = gy.shape
    if (Ho, Wo) != ((H - 1) // stride + 1, (W - 1) // stride + 1):
        raise RuntimeError(f"paradis::geocyclic_avgpool5_backward: grad_y {tuple(gy.shape)} does not match an "
                           f"input of {H} x {W} with stride {stride}")
    native = _geo_bf16(gy)
    gs = gy.contiguous() if native else gy.float().contiguous()
    gx = torch.empty((B, Cn, H, W), dtype=gs.dtype, device=gy.device)
    name = "paradis_geocyclic_avgpool5_bwd_bf16" if native else "paradis_geocyclic_avgpool5_bwd"
    with torch.cuda.device(gy.device):
        rc = getattr(_lib.lib(), name)(_ptr(gs), _ptr(gx), B, Cn, H, W, stride, _stream(gy))
    _lib.check(rc, name)
    return gx.to(gy.dtype)


@_geocyclic_avgpool5_backward.register_fake
def _(gy, H, W, stride):
    return gy.new_empty((gy.shape[0], gy.shape[1], H, W))


def _pool_setup(ctx, inputs, output):
    x, stride = inputs
    ctx.stride, ctx.shape, ctx.dtype = stride, tuple(x.shape), x.dtype


def _pool_backward(ctx, gy):
    _no_fwd_over_rev(gy)
    B, Cn, H, W = ctx.shape
    return torch.ops.paradis.geocyclic_avgpool5_backward(gy, H, W, ctx.stride).to(ctx.dtype), None


_geocyclic_avgpool5.register_autograd(_pool_backward, setup_context=_pool_setup)


class _PoolFn(torch.autograd.Function):
    """paradis::geocyclic_avgpool5 with a jvp rule: the op is linear, its tangent is the op applied to the tangent."""

    @staticmethod
    def forward(x, stride):
        return torch.ops.paradis.geocyclic_avgpool5(x, stride)

    setup_context = staticmethod(_pool_setup)
    backward = staticmethod(_pool_backward)
    vmap = staticmethod(_no_vmap)

    @staticmethod
    def jvp(ctx, dx, _):
        return torch.ops.paradis.geocyclic_avgpool5(dx, ctx.stride)


def geocyclic_avgpool5(x: Tensor, stride: int) -> Tensor:
    """``AvgPool2d(5, stride)(GeoCyclicPadding(2)(x))`` (model/blocks.py:57-71) in one kernel."""
    assert x.dim() == 4, "Input must be 4-dimensional [batch, channels, lat, lon]"
    assert x.shape[3] % 2 == 0, "Number of longitude points must be even"
    if _tangent_path(x):
        return _PoolFn.apply(x, int(stride))
    return torch.ops.paradis.geocyclic_avgpool5(x, int(stride))


# --------------------------------------------------------------------------------------
# halo_pack: boundary rows of the band tensors into the symmetric-memory outbox (halo.PeerHalo), one launch
# --------------------------------------------------------------------------------------
@torch.library.custom_op("paradis::halo_pack", mutates_args=("box",), device_types="cuda")
def _halo_pack(xs: List[Tensor], box: Tensor, h: int) -> None:
    import ctypes as C
    n = len(xs)
    B, V, rows, W = xs[0].shape
    for t in xs:
        if (t.dtype != torch.float32 or tuple(t.shape) != (B, V, rows, W) or t.stride(3) != 1 or t.stride(2) != W
                or t.stride(1) != rows * W):
            raise RuntimeError("halo_pack expects fp32 [B, V, rows, W] tensors whose inner three dims are contiguous")
    if box.dtype != torch.float32 or not box.is_contiguous() or box.numel() < n * 2 * B * V * h * W:
        raise RuntimeError("halo_pack: outbox too small or not contiguous fp32")
    src = (C.c_void_p * n)(*[t.data_ptr() for t in xs])
    sB = (C.c_int64 * n)(*[t.stride(0) if B > 1 else V * rows * W for t in xs])
    with torch.cuda.device(box.device):
        rc = _lib.lib().paradis_halo_pack(src, sB, n, B, V, rows, W, h, _ptr(box), _stream(box))
    _lib.check(rc, "paradis_halo_pack")


def halo_pack(xs: List[Tensor], box: Tensor, h: int) -> None:
    """First and last `h` rows of every tensor of `xs` ([B, V, rows, W]) -> box[len(xs)][2][B*V][h][W]."""
    torch.ops.paradis.halo_pack(list(xs), box, int(h))


def geocyclic_dwconv(x: Tensor, weight: Tensor, bias: Optional[Tensor] = None) -> Tensor:
    """``depthwise_conv(GeoCyclicPadding((k-1)//2)(x))`` in one kernel (k = 3, 5, 7): drop-in for the first
    two lines of SepConv.forward (model/blocks.py:112-114).  Differentiable w.r.t. x, weight and bias."""
    assert x.dim() == 4, "Input must be 4-dimensional [batch, channels, lat, lon]"
    assert x.shape[3] % 2 == 0, "Number of longitude points must be even"
    if _tangent_path(x, weight, bias):
        return _DwConvFn.apply(x, weight, bias)
    return torch.ops.paradis.geocyclic_dwconv(x, weight, bias)


# --------------------------------------------------------------------------------------
# host-buffer entry (end-to-end measurement path)
# --------------------------------------------------------------------------------------
def host_fwd_bwd(geometry: SLGeometry, h_field: Tensor, h_u: Tensor, h_v: Tensor, h_grad_out: Tensor,
                 h_out: Tensor, h_gfield: Tensor, h_gu: Tensor, h_gv: Tensor, dt: float,
                 interpolation: str = "bilinear", pole_fix: bool = True, math: str = "fast",
                 chunk_planes: int = 8, scratch: Tensor | None = None,
                 cfl_cells: float = DEFAULT_CFL_CELLS) -> Tensor:
    """Forward + backward with HOST tensors (pinned recommended) through
    ``paradis_sl_advect_fwd_bwd_host``: chunked, H2D / kernels / D2H overlapped inside the
    library; returns (and reuses) the device scratch buffer."""
    L = _lib.lib()
    B, V, H, W = h_field.shape
    for t in (h_field, h_u, h_v, h_grad_out, h_out, h_gfield, h_gu, h_gv):
        if t.is_cuda or t.dtype != torch.float32 or not t.is_contiguous() or tuple(t.shape) != (B, V, H, W):
            raise RuntimeError("host_fwd_bwd expects contiguous fp32 CPU tensors of one shape")
    dev = geometry.tables.device
    need = L.paradis_sl_host_scratch_bytes(H, W, chunk_planes)
    if scratch is None or scratch.numel() < need:
        scratch = torch.empty(need, dtype=torch.uint8, device=dev)
    g = _geom_struct(geometry.tables, geometry.scalars, geometry.windows)
    torch.cuda.current_stream(dev).synchronize()  # the library runs on its own streams
    with torch.cuda.device(dev):
        rc = L.paradis_sl_advect_fwd_bwd_host(C.byref(g), _ptr(h_field), _ptr(h_u), _ptr(h_v), _ptr(h_grad_out),
                                              _ptr(h_out), _ptr(h_gfield), _ptr(h_gu), _ptr(h_gv), B * V, dt,
                                              _lib.INTERP[interpolation], int(pole_fix), _lib.MATH[math],
                                              float(cfl_cells), chunk_planes, _ptr(scratch), scratch.numel())
    _lib.check(rc, "paradis_sl_advect_fwd_bwd_host")
    return scratch


# --------------------------------------------------------------------------------------
# low-level access for measurement: backward phases separately, caller-held buffers
# --------------------------------------------------------------------------------------
class RawAdvection:
    """Pre-allocated buffers + direct C-ABI calls (no autograd, no allocation per call).
    Used by bench.py to time forward, backward-arrival and backward-gather separately."""

    def __init__(self, geometry: SLGeometry, B: int, V: int, interpolation="bilinear", pole_fix=True, math="fast",
                 cfl_cells: float = DEFAULT_CFL_CELLS):
        self.geo, self.B, self.V, self.cfl = geometry, B, V, float(cfl_cells)
        self.interp, self.pole_fix, self.math = _lib.INTERP[interpolation], int(pole_fix), _lib.MATH[math]
        dev = geometry.tables.device
        L = _lib.lib()
        H, W, own0, ownN, arr0, arrN, fld0, fldN = geometry.windows[:8]
        self.out = torch.empty((B, V, ownN, W), dtype=torch.float32, device=dev)
        self.gfield, self.gu, self.gv = [torch.empty_like(self.out) for _ in range(3)]
        self.ws_f = torch.empty(L.paradis_sl_advect_fwd_workspace(B, V), dtype=torch.uint8, device=dev)
        self.ws_b = torch.empty(L.paradis_sl_advect_bwd_workspace(B, V, arrN, W), dtype=torch.uint8, device=dev)
        self.g = _geom_struct(geometry.tables, geometry.scalars, geometry.windows)
        self.status = _status_word(dev)

    def forward(self, field, u, v, dt):
        rc = _lib.lib().paradis_sl_advect_fwd(C.byref(self.g), _ptr(field), _ptr(u), _ptr(v), _ptr(self.out), self.B,
                                              self.V, field.stride(0), u.stride(0), v.stride(0), dt, self.interp,
                                              self.pole_fix, self.math, _ptr(self.ws_f), self.ws_f.numel(),
                                              _ptr(self.status), _stream(field))
        _lib.check(rc, "paradis_sl_advect_fwd")
        return self.out

    def backward(self, grad_out, field, u, v, dt, phases=3):
        rc = _lib.lib().paradis_sl_advect_bwd(C.byref(self.g), _ptr(grad_out), _ptr(field), _ptr(u), _ptr(v),
                                              _ptr(self.gfield), _ptr(self.gu), _ptr(self.gv), self.B, self.V,
                                              grad_out.stride(0), field.stride(0), u.stride(0), v.stride(0), dt,
                                              self.interp, self.pole_fix, self.math, phases, self.cfl, _ptr(self.ws_b),
                                              self.ws_b.numel(), _ptr(self.status), _stream(field))
        _lib.check(rc, "paradis_sl_advect_bwd")
        return self.gfield, self.gu, self.gv


def departure_coords(u: Tensor, v: Tensor, geometry: SLGeometry, dt: float, interpolation="bilinear",
                     math="fast") -> Tensor:
    """Parity instrument: [B, V, 11, H, W] = (ix, iy, sin lat', cos lat', sin lon', cos lon', sin_lat, num, den, lat, lon),
    the intermediates of model/advection.py:82-94 and the sampler coordinates ATen floors."""
    L = _lib.lib()
    u, v = _inner_contig(u.float()), _inner_contig(v.float())
    B, V, R, W = u.shape
    out = torch.empty((B, V, 11, geometry.windows[3], W), dtype=torch.float32, device=u.device)
    g = _geom_struct(geometry.tables, geometry.scalars, geometry.windows)
    with torch.cuda.device(u.device):
        rc = L.paradis_sl_departure_coords(C.byref(g), _ptr(u), _ptr(v), _ptr(out), B, V, u.stride(0), v.stride(0),
                                           dt, _lib.INTERP[interpolation], _lib.MATH[math], _stream(u))
    _lib.check(rc, "paradis_sl_departure_coords")
    return out
