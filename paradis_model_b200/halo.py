"""Latitude-band decomposition of one 0.25-degree field across GPUs (SURVEY 8e).

Rank k of G owns a contiguous band of full longitude circles.  Because every band holds whole
circles, the longitude wrap and the 180-degree pole shift of the GeoCyclic map stay local; the pole
reflection rows and the pole-mean rows belong to the first / last band.  The only exchange is with
the two latitude neighbours:

  forward : `halo` rows of `field` either side (departure stencils reach at most cfl + stencil rows)
  backward: `halo` rows of (grad_out, u, v) either side, so that every band computes its own
            grad_field rows with the deterministic inverse-stencil gather -- one exchange, no
            reverse add, bit-identical to the single-GPU result for the general path.

Two transports:

* `exchange_rows`: point-to-point `torch.distributed.batch_isend_irecv` (NCCL send/recv over NVLink
  on GPUs, gloo in the CPU tests) into an assembled [lo + rows + hi] tensor.
* `PeerHalo` (field halos, GPUs only): every rank publishes its boundary rows in a symmetric-memory
  outbox; the neighbours' outboxes are mapped into this process and their addresses are handed to
  the kernels (`paradis_sl_geom.fld_peer_lo/hi`), which load the stencil taps that fall outside the
  band straight from the peer GPU over NVLink -- the halo exchange is fused into the gather, nothing
  is assembled or copied on the receiving side.

There is no collective on the data path.  The reference has no spatial decomposition at all (its
only parallelism is DDP, train.py:49); this module is new.
"""
from __future__ import annotations

import math
from dataclasses import dataclass
from typing import List, Optional, Tuple

import torch
import torch.distributed as dist

STENCIL_ROWS = {"bilinear": 2, "bicubic": 4}


@dataclass
class BandPlan:
    H: int
    W: int
    rank: int
    world: int
    row0: int          # first owned row (global)
    rows: int          # owned rows
    halo: int          # rows exchanged with each neighbour
    lo: int            # rows received from the southern neighbour (0 for the first band)
    hi: int            # rows received from the northern neighbour (0 for the last band)

    @property
    def ext_row0(self) -> int:
        return self.row0 - self.lo

    @property
    def ext_rows(self) -> int:
        return self.lo + self.rows + self.hi

    def windows(self) -> Tuple[Tuple[int, int], Tuple[int, int]]:
        """(own, ext) as (row0, rows) pairs for SLGeometry.band()."""
        return (self.row0, self.rows), (self.ext_row0, self.ext_rows)


def band_rows(H: int, world: int, cost: Optional[List[float]] = None, overhead_rows: float = 0.0,
              min_rows: int = 1) -> List[Tuple[int, int]]:
    """Split H rows into `world` contiguous bands: equal height, or -- when a per-row `cost` is given (rows near the
    poles are several times more expensive in the backward, see `row_costs`) -- the split that levels the bands'
    costs (dynamic programme over the cut rows), a band of n rows costing  sum(cost) * (1 + overhead_rows / n):  every CTA segment of the row
    sweep re-plays ring - 1 arrival rows before its first own row, at the latitude it works at, so a band carries
    a number of extra rows that does not shrink with its height (tools/band_local.py measures it)."""
    if cost is None:
        base, rem = divmod(H, world)
        out, r = [], 0
        for k in range(world):
            n = base + (1 if k < rem else 0)
            out.append((r, n))
            r += n
        return out
    import numpy as np
    S = np.concatenate([[0.0], np.cumsum(np.asarray(cost, dtype=np.float64))])
    a = np.arange(H + 1)[:, None]
    b = np.arange(H + 1)[None, :]
    n = b - a
    with np.errstate(divide="ignore", invalid="ignore"):
        C = np.where(n >= max(min_rows, 1), (S[b] - S[a]) * (1.0 + overhead_rows / np.maximum(n, 1)), np.inf)
    # sum of 8th powers instead of the plain maximum: the same most expensive band to within a row, and the other
    # bands come out balanced among themselves too (a pure min-max leaves them arbitrary)
    C = (C / C[0, H]) ** 8
    dp = C[0].copy()                                  # one band covering rows [0, b)
    arg = []
    for _ in range(1, world):
        M = dp[:, None] + C                           # band [a, b) after the best split of [0, a)
        arg.append(M.argmin(axis=0))
        dp = M.min(axis=0)
    if not np.isfinite(dp[H]):
        raise ValueError(f"{H} rows cannot be split into {world} bands of at least {min_rows} rows")
    cuts, e = [H], H
    for k in range(world - 2, -1, -1):
        e = int(arg[k][e])
        cuts.append(e)
    cuts.append(0)
    cuts = cuts[::-1]
    return [(cuts[k], cuts[k + 1] - cuts[k]) for k in range(world)]


def row_costs(H: int, W: int, cfl_cells: float, strip: int = 240, base: float = None) -> List[float]:
    """Relative backward cost of a row on a pole-to-pole mesh, the model the row-sweep kernel balances its own CTAs
    with (csrc/paradis_sl.cu, launch_rows): a constant for the producers plus the number of 32-record steps a
    consumer scans for the row -- its strip plus the longitudinal reach of the row either side, which grows as
    1 / cos(lat) and becomes the whole circle next to the poles."""
    if base is None:      # the forward and the producers: about 2.5 scan steps' worth of time per row at C3
        base = 2.5
    dphi = math.pi / max(H - 1, 1)
    delta = cfl_cells * dphi
    out = []
    for i in range(H):
        lat = abs(-math.pi / 2 + i * dphi) + delta
        cells = W
        if lat < math.pi / 2 - 1e-9:
            sdl = math.sin(delta) / math.cos(lat)
            if sdl < 1.0:
                cells = min(W, math.asin(sdl) / (2 * math.pi / W) + 4)
        scan = min(W, strip + 2 * cells)
        out.append(base + math.ceil(scan / 32))
    return out


def halo_rows(cfl_cells: float, interpolation: str) -> int:
    """Rows a departure stencil can reach beyond its arrival row: ceil(cfl) for the trajectory plus
    the stencil extent (and one row of slack for the floor)."""
    return int(math.ceil(cfl_cells)) + STENCIL_ROWS[interpolation] + 1


def make_plan(H: int, W: int, rank: int, world: int, cfl_cells: float, interpolation: str = "bilinear",
              balance: bool = False) -> BandPlan:
    """`balance=True` sizes the bands by backward cost instead of by height (fewer rows for the ranks
    that own a polar cap)."""
    halo = halo_rows(cfl_cells, interpolation)
    if balance and world > 1:
        # (CTAs + planes) / planes segments per plane, each re-playing ring - 1 = 2 ceil(cfl) + stencil rows - 1 rows
        warm = 3.0 * (2 * math.ceil(cfl_cells) + STENCIL_ROWS[interpolation] - 1)
        try:
            bands = band_rows(H, world, row_costs(H, W, cfl_cells), warm, halo + 1)
        except ValueError:
            bands = band_rows(H, world)
    else:
        bands = band_rows(H, world)
    row0, rows = bands[rank]
    if world > 1 and min(n for _, n in bands) <= halo:   # strictly thicker: a pole row is never in a neighbour's halo
        raise ValueError(f"bands of {min(n for _, n in bands)} rows are not thicker than the halo ({halo} rows): "
                         "use fewer ranks or a smaller cfl_cells")
    lo = halo if rank > 0 else 0
    hi = halo if rank < world - 1 else 0
    return BandPlan(H, W, rank, world, row0, rows, halo, lo, hi)


def exchange_rows_multi(xs: List[torch.Tensor], plan: BandPlan, group=None) -> List[torch.Tensor]:
    """Each x: [B, C, rows, W] owned rows -> [B, C, lo + rows + hi, W] with the neighbours' boundary rows.

    All sends and receives of all tensors go out as ONE batch (NCCL groups them into one launch); every
    tensor is copied exactly once (into the interior of its extended buffer)."""
    if plan.world == 1:
        return list(xs)
    h, ops, exts, keep = plan.halo, [], [], []
    for x in xs:
        B, C, n, W = x.shape
        assert n == plan.rows and W == plan.W
        ext = x.new_empty((B, C, plan.ext_rows, W))
        ext[:, :, plan.lo:plan.lo + n] = x
        exts.append(ext)
        if plan.rank > 0:                                   # southern neighbour
            send = x[:, :, :h].contiguous()
            recv = x.new_empty((B, C, h, W))
            ops += [dist.P2POp(dist.isend, send, plan.rank - 1, group),
                    dist.P2POp(dist.irecv, recv, plan.rank - 1, group)]
            keep.append((ext, "lo", recv, n))
        if plan.rank < plan.world - 1:                      # northern neighbour
            send = x[:, :, n - h:].contiguous()
            recv = x.new_empty((B, C, h, W))
            ops += [dist.P2POp(dist.isend, send, plan.rank + 1, group),
                    dist.P2POp(dist.irecv, recv, plan.rank + 1, group)]
            keep.append((ext, "hi", recv, n))
    for req in dist.batch_isend_irecv(ops):
        req.wait()
    for ext, side, recv, n in keep:
        if side == "lo":
            ext[:, :, :plan.lo] = recv
        else:
            ext[:, :, plan.lo + n:] = recv
    return exts


def exchange_rows(x: torch.Tensor, plan: BandPlan, group=None) -> torch.Tensor:
    """Single-tensor form of :func:`exchange_rows_multi`."""
    return exchange_rows_multi([x], plan, group)[0]


class PeerHalo:
    """Boundary rows of the band tensors published in NVLink peer memory (torch symmetric memory).

    box[parity][slot][side]: side 0 = this band's first `halo` rows (read by the southern neighbour as ITS northern
    halo), side 1 = its last `halo` rows (read by the northern neighbour as its southern halo); slot 0 = field,
    slots 1..3 = u, v, grad_out of the backward.  A publish is stream-ordered device work: ONE pack kernel
    (`paradis_halo_pack`) into the outbox of the current parity, then ONE barrier (everybody's rows are in place);
    the kernels then dereference `lo` / `hi` -- addresses inside the NEIGHBOURS' outboxes -- directly.

    The outbox is double-buffered so that no barrier is needed BEFORE the pack: publish n + 2 overwrites the buffer
    of publish n, and a rank only gets there after passing the barrier of publish n + 1, which every neighbour
    reaches after its kernels that read publish n (same stream).  Every rank must publish the same sequence."""

    def __init__(self, plan: BandPlan, B: int, V: int, device, group=None, pull_field: bool = False,
                 pull_all: bool = False):
        import torch.distributed._symmetric_memory as symm
        self.plan, self.planes = plan, B * V
        h, W = plan.halo, plan.W
        self.box = symm.empty((2, 4, 2, B * V, h, W), dtype=torch.float32, device=device)
        self.hdl = symm.rendezvous(self.box, group=group if group is not None else dist.group.WORLD)
        side_elems = B * V * h * W
        side_bytes = side_elems * 4
        self._side_elems = side_elems
        ptrs = self.hdl.buffer_ptrs
        south = int(ptrs[plan.rank - 1]) if plan.rank > 0 else 0
        north = int(ptrs[plan.rank + 1]) if plan.rank < plan.world - 1 else 0
        # my southern halo = the southern neighbour's LAST rows (its side 1); northern halo = side 0 of the northern one
        self._lo = [[south + ((8 * par) + 2 * k + 1) * side_bytes if south else 0 for k in range(4)] for par in range(2)]
        self._hi = [[north + ((8 * par) + 2 * k) * side_bytes if north else 0 for k in range(4)] for par in range(2)]
        self.parity = 1                       # parity of the LAST publish (the first one uses 0)
        # pull_field / pull_all: the halo rows (of `field` only / of all published tensors) are PULLED into local memory
        # right after the publish barrier -- one strided peer-memory copy per side over NVLink, no NCCL -- instead of
        # being read in place by the stencil taps and the TMA bulk copies of the kernels.  Thick bands (N=2) are faster
        # in place (the copies cost more than the remote accesses they save); thin bands pay relatively more for the
        # NVLink latency inside the kernels.  See DESIGN section 5 for the measurements.
        self.local = None
        self._peer_views = None
        self._pull_slots = 4 if pull_all else (1 if pull_field else 0)
        if self._pull_slots:
            ns = self._pull_slots
            self.local = torch.empty((2, 4, B * V, h, W), dtype=torch.float32, device=device)   # [side][slot]
            full = (2, 4, 2, B * V, h, W)
            views = []
            for par in range(2):
                lo_v = self.hdl.get_buffer(plan.rank - 1, full, torch.float32, 0)[par, :, 1] if south else None
                hi_v = self.hdl.get_buffer(plan.rank + 1, full, torch.float32, 0)[par, :, 0] if north else None
                views.append((lo_v, hi_v))
            self._peer_views = views
            loc = [[self.local[sd, k].data_ptr() for k in range(4)] for sd in range(2)]
            self._lo_local = [loc[0][k] if (south and k < ns) else None for k in range(4)]
            self._hi_local = [loc[1][k] if (north and k < ns) else None for k in range(4)]

    @property
    def lo(self):
        """Addresses of this band's southern halo rows, one per slot: inside the neighbour's outbox, or local if pulled."""
        p = self._lo[self.parity]
        if self.local is None:
            return p
        return [self._lo_local[k] if self._lo_local[k] is not None else p[k] for k in range(4)]

    @property
    def hi(self):
        p = self._hi[self.parity]
        if self.local is None:
            return p
        return [self._hi_local[k] if self._hi_local[k] is not None else p[k] for k in range(4)]

    def _publish(self, tensors) -> None:
        from .ops import halo_pack
        t0 = tensors[0]
        assert t0.shape[2] == self.plan.rows and t0.shape[0] * t0.shape[1] == self.planes
        self.parity ^= 1
        halo_pack([t if t.stride(3) == 1 and t.stride(2) == t.shape[3] and t.stride(1) == t.shape[2] * t.shape[3]
                   else t.contiguous() for t in tensors], self.box[self.parity], self.plan.halo)
        self.hdl.barrier(channel=0)
        if self.local is not None:
            n = min(len(tensors), self._pull_slots)            # slots this publish filled (1: field, 4: backward)
            for sd, view in enumerate(self._peer_views[self.parity]):
                if view is not None:
                    self.local[sd, :n].copy_(view[:n])

    def publish(self, field: torch.Tensor) -> None:
        self._publish([field])

    def publish_backward(self, field: torch.Tensor, u: torch.Tensor, v: torch.Tensor, g: torch.Tensor) -> None:
        """One pack and one barrier for all four tensors of the backward."""
        self._publish([field, u, v, g])

    def peer(self):
        return (self.lo[0], self.hi[0], self.plan.halo)

    def arr_peer(self):
        return (self.lo[1:4], self.hi[1:4], self.plan.halo)


class _LatBandFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, field, u, v, geometry, plan, dt, interp, pole_fix, math, cfl, group, peer):
        from . import _lib
        own, ext = plan.windows()
        if peer is not None:                 # field halo read in place from the neighbours (fused exchange)
            field = field.contiguous()
            peer.publish(field)
            g = geometry.band(own, own, own, peer.peer())
            f_saved = field
        else:
            f_saved = exchange_rows(field, plan, group)
            g = geometry.band(own, own, ext)
        out = torch.ops.paradis.sl_advect(f_saved, u, v, g.tables, g.scalars, dt, _lib.INTERP[interp], pole_fix,
                                          _lib.MATH[math], g.windows, cfl)
        ctx.save_for_backward(f_saved, u, v)
        ctx.meta = (geometry, plan, dt, interp, pole_fix, math, cfl, group, peer)
        return out

    @staticmethod
    def backward(ctx, grad_out):
        from . import _lib
        f_saved, u, v = ctx.saved_tensors
        geometry, plan, dt, interp, pole_fix, math, cfl, group, peer = ctx.meta
        own, ext = plan.windows()
        if peer is not None:
            # nothing is exchanged or assembled: all four tensors keep their own rows, the kernels read the
            # neighbours' boundary rows in place (the outboxes may have been reused since forward: republish)
            g_ext, u_ext, v_ext = grad_out.contiguous(), u.contiguous(), v.contiguous()
            peer.publish_backward(f_saved, u_ext, v_ext, g_ext)
            g = geometry.band(own, ext, own, peer.peer(), peer.arr_peer())
        else:
            g_ext, u_ext, v_ext = exchange_rows_multi([grad_out.contiguous(), u, v], plan, group)   # one NCCL group
            g = geometry.band(own, ext, ext)
        gf, gu, gv = torch.ops.paradis.sl_advect_backward(g_ext, f_saved, u_ext, v_ext, g.tables, g.scalars, dt,
                                                          _lib.INTERP[interp], pole_fix, _lib.MATH[math], g.windows,
                                                          cfl, True, True)
        return gf, gu, gv, None, None, None, None, None, None, None, None, None


class BandKernels:
    """The raw (no autograd, preallocated) forward / backward of one band, one pair per outbox parity: the peer
    addresses a kernel reads depend on which half of the double-buffered outbox the last publish filled."""

    def __init__(self, geometry, plan: BandPlan, peer: "PeerHalo", B: int, V: int, interp: str, math: str, cfl: float):
        self.args = (geometry, plan, peer, B, V, interp, math, cfl)
        self._k = {}

    def _get(self, kind: str):
        from .ops import RawAdvection
        geometry, plan, peer, B, V, interp, math, cfl = self.args
        key = (kind, peer.parity)
        if key not in self._k:
            own, ext = plan.windows()
            g = (geometry.band(own, own, own, peer.peer()) if kind == "f"
                 else geometry.band(own, ext, own, peer.peer(), peer.arr_peer()))
            self._k[key] = RawAdvection(g, B, V, interp, True, math, cfl)
        return self._k[key]

    def forward(self, field, u, v, dt):
        return self._get("f").forward(field, u, v, dt)

    def backward(self, go, field, u, v, dt, phases=3):
        return self._get("b").backward(go, field, u, v, dt, phases)


def lat_band_advect(field, u, v, geometry, plan: BandPlan, dt: float, interpolation="bilinear", pole_fix=True,
                    math="fast", cfl_cells: float = 8.0, group=None, peer: Optional["PeerHalo"] = None):
    """sl_advect on this rank's latitude band: field, u, v, result are [B, V, plan.rows, W].

    `cfl_cells` sizes the halo (plan.halo must have been built with the same value): unlike the
    single-GPU call it is a CONTRACT here -- a departure stencil that leaves the halo sets the
    device status word (paradis_model_b200.check_status raises DISPLACEMENT).  With `peer` (a PeerHalo
    built for the same plan and plane count) the field halo is not exchanged at all: the kernels read
    the neighbours' boundary rows in place over NVLink."""
    return _LatBandFn.apply(field, u, v, geometry, plan, float(dt), interpolation, bool(pole_fix), math,
                            float(cfl_cells), group, peer)


# ------------------------------------------------------------------------------------------
# strong-scaling benchmark leg (bench.py --decomp latband)
# ------------------------------------------------------------------------------------------
def bench_latband(args, workload, rank, world, dev):
    import json
    import paradis_model_b200 as P
    from . import synthetic as S
    from bench import BYTES_STEP, CFL_CELLS, measured_peak   # only reached from bench.py --decomp latband

    H, W, V, Bg, poles = workload
    dt = S.DT_DEFAULT
    lat, lon = S.make_grids(H, W, poles)
    geo = P.SLGeometry.from_grids(lat.to(dev), lon.to(dev))
    plan = make_plan(H, W, rank, world, CFL_CELLS, args.interp, balance=poles)
    # every rank draws the same global tensors (same seed) and keeps its band: the global problem is
    # identical for every N (strong scaling)
    full = S.white_noise_inputs(H, W, Bg, V, dt, seed=0)
    sl = slice(plan.row0, plan.row0 + plan.rows)
    field, u, v, go = [t[:, :, sl].contiguous().to(dev) for t in full]
    del full
    peer, transport = None, "NCCL send/recv for field, grad_out, u, v"
    if not getattr(args, "no_p2p", False):
        try:
            peer = PeerHalo(plan, Bg, V, dev, pull_field=getattr(args, "pull_field", False),
                            pull_all=getattr(args, "pull_all", False))
            if getattr(args, "pull_all", False):
                transport = ("halos over NVLink peer memory (symmetric memory), no NCCL on the data path: the boundary rows of field, "
                             "u, v, grad_out are pulled into local buffers by one strided peer copy per side after the publish barrier")
            else:
                transport = ("halos over NVLink peer memory (symmetric memory), no NCCL on the data path: u, v, grad_out rows streamed in "
                             "place by TMA bulk copies inside the backward kernel, field rows "
                             + ("pulled into a local buffer by one peer copy per side after the publish barrier"
                                if getattr(args, "pull_field", False) else "read in place by the stencil taps"))
        except Exception as exc:   # symmetric memory unavailable: NCCL transport for everything
            transport += f" (symmetric memory unavailable: {type(exc).__name__})"

    def step():
        f = field.requires_grad_(True)
        uu, vv = u.requires_grad_(True), v.requires_grad_(True)
        out = lat_band_advect(f, uu, vv, geo, plan, dt, args.interp, True, args.math, CFL_CELLS, None, peer)
        out.backward(go)
        f.grad = uu.grad = vv.grad = None

    mode = "eager autograd (torch.library op)"
    if peer is not None and not getattr(args, "no_graph", False):
        # The whole step -- publish, forward, publish, fused backward with its side streams and the
        # symmetric-memory barriers -- is stream-ordered device work: capture it once in a CUDA graph and
        # replay it, which removes the host launch overhead that dominates thin bands.
        try:
            K = BandKernels(geo, plan, peer, Bg, V, args.interp, args.math, CFL_CELLS)

            def raw_step():                 # two publishes: the outbox parity is the same at the start of every step
                peer.publish(field)
                K.forward(field, u, v, dt)
                peer.publish_backward(field, u, v, go)
                K.backward(go, field, u, v, dt, 3)

            for _ in range(3):
                raw_step()
            torch.cuda.synchronize()
            dist.barrier()
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                raw_step()
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            dist.barrier()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                raw_step()
            step = graph.replay
            mode = "one CUDA graph per step (C-ABI calls + symmetric-memory barriers captured)"
        except Exception as exc:
            mode += f" (graph capture unavailable: {type(exc).__name__}: {exc})"[:200]

    from bench import BYTES_FWD, BYTES_BWD, ClockSampler
    for _ in range(max(3, args.warmup)):
        step()
    torch.cuda.synchronize()
    dist.barrier()
    sampler = ClockSampler(dev.index if dev.index is not None else 0)
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        step()
    e1.record()
    torch.cuda.synchronize()
    clocks = sampler.stop()
    dist.barrier()
    P.check_status(dev)
    t = torch.tensor([e0.elapsed_time(e1)], device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_step = float(t.item()) / args.steps

    # ---- the two phases of a band, timed separately on every rank (eager C-ABI calls; max over ranks)
    if peer is not None:
        K2 = BandKernels(geo, plan, peer, Bg, V, args.interp, args.math, CFL_CELLS)
        phase = []
        for fn, pub in ((lambda: K2.forward(field, u, v, dt), lambda: peer.publish(field)),
                        (lambda: K2.backward(go, field, u, v, dt, 3), lambda: peer.publish_backward(field, u, v, go))):
            for _ in range(4):                           # both outbox parities warm (kernel objects are built lazily)
                pub(); fn()
            torch.cuda.synchronize(); dist.barrier()
            n_ph = max(3, min(args.steps, 10))
            acc = 0.0
            for _ in range(n_ph):
                pub()                                    # publishes and barriers outside the timed kernel phase
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record(); fn(); b.record()
                torch.cuda.synchronize()
                acc += a.elapsed_time(b)
            tp = torch.tensor([acc / n_ph], device=dev)
            dist.all_reduce(tp, op=dist.ReduceOp.MAX)
            phase.append(float(tp.item()))
    else:
        phase = [float("nan"), float("nan")]

    # ---- end to end through the public API: pinned host bands -> H2D -> lat_band_advect fwd + bwd -> D2H
    e2e = None
    if not getattr(args, "no_e2e", False):
        h_in = [t.cpu().pin_memory() for t in (field, u, v, go)]
        h_out = [torch.empty_like(h_in[0]).pin_memory() for _ in range(4)]

        def e2e_step():
            f, uu, vv, g = [t.to(dev, non_blocking=True) for t in h_in]
            f.requires_grad_(True); uu.requires_grad_(True); vv.requires_grad_(True)
            out = lat_band_advect(f, uu, vv, geo, plan, dt, args.interp, True, args.math, CFL_CELLS, None, peer)
            out.backward(g)
            for dst, src in zip(h_out, (out.detach(), f.grad, uu.grad, vv.grad)):
                dst.copy_(src, non_blocking=True)
            torch.cuda.synchronize()

        e2e_step()
        dist.barrier()
        n_e2e = max(2, min(args.steps, 5))
        import time as _time
        t0 = _time.perf_counter()
        for _ in range(n_e2e):
            e2e_step()
        te = torch.tensor([(_time.perf_counter() - t0) / n_e2e], device=dev)
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
        band_bytes = torch.tensor([4 * field.numel() * 4], device=dev, dtype=torch.float64)
        dist.all_reduce(band_bytes)
        e2e = {"value": Bg * V * H * W / float(te.item()), "unit": "grid-pt*ch/s",
               "h2d_bytes_per_step": int(band_bytes.item()), "d2h_bytes_per_step": int(band_bytes.item()),
               "ms_per_step": float(te.item()) * 1e3, "steps": n_e2e,
               "api": "paradis_model_b200.halo.lat_band_advect (autograd) on pinned host bands, all ranks, bytes summed over ranks"}

    # ---- the communication-free alternative in the same run: every rank a full replica (batch-sharded, weak scaling)
    batch = None
    if not getattr(args, "no_batch", False):
        full_d = [t.to(dev) for t in S.white_noise_inputs(H, W, Bg, V, dt, seed=rank)]
        from .ops import RawAdvection
        Rr = RawAdvection(geo, Bg, V, args.interp, True, args.math, CFL_CELLS)

        def rstep():
            Rr.forward(full_d[0], full_d[1], full_d[2], dt)
            Rr.backward(full_d[3], full_d[0], full_d[1], full_d[2], dt, 3)

        for _ in range(3):
            rstep()
        torch.cuda.synchronize(); dist.barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        nb = max(3, min(args.steps, 20))
        a.record()
        for _ in range(nb):
            rstep()
        b.record()
        torch.cuda.synchronize(); dist.barrier()
        tb = torch.tensor([a.elapsed_time(b) / nb], device=dev)
        dist.all_reduce(tb, op=dist.ReduceOp.MAX)
        batch = {"value": world * Bg * V * H * W / (float(tb.item()) * 1e-3), "unit": "grid-pt*ch/s",
                 "ms_per_step": float(tb.item()), "scaling": "weak",
                 "parallelism": f"batch-sharded x{world}: one full {H}x{W} replica per GPU, no communication"}
        del full_d, Rr

    if rank == 0:
        pts = Bg * V * H * W
        peak, src = measured_peak()
        gbs = BYTES_STEP * pts / (ms_step * 1e-3) / 1e9
        halo_bytes = 2 * plan.halo * W * V * Bg * 4
        dom = 1 if not (phase[1] != phase[1]) and phase[1] >= phase[0] else 0
        names = ["sl_fwd_kernel", "sl_bwd_rows_kernel" if args.interp == "bilinear" else "sl_bwd_sweep_kernel"]
        alg = [BYTES_FWD, BYTES_BWD]
        band_pts = pts / world                                   # max-over-ranks time against the mean band
        ach = alg[dom] * band_pts / (phase[dom] * 1e-3) / 1e9 if phase[dom] == phase[dom] else None
        line = {
            "metric": "SL advection fwd+bwd grid-pts*ch/s", "value": pts / (ms_step * 1e-3), "unit": "grid-pt*ch/s",
            "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": ms_step,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"{args.workload}: {H}x{W} mesh, V={V}, batch {Bg} GLOBAL (the N=1 problem), {args.interp}, "
                                   f"math={args.math}, pole_fix, cfl_cells={CFL_CELLS}, latitude bands x{world}, halo {plan.halo} rows",
                       "inputs": "field~N(0,1); u,v~N(0,(2 cells)^2) clipped at +-4 cells; grad_out~N(0,1); seed 0, same global tensors for every N",
                       "l2": "per-rank inputs exceed the 126 MB L2 up to N=8 (133 MB per rank there); no flush",
                       "parallelism": f"latband{world} (cost-balanced bands, rank 0 owns {plan.rows} rows): {transport}; "
                                      f"{halo_bytes} B of halo per rank per tensor",
                       "launch": mode},
            "roofline": {"bound": "hbm", "kernel": names[dom], "achieved": ach, "peak": peak, "unit": "GB/s",
                         "frac": (ach / peak) if ach else None, "traffic": None, "peak_source": src,
                         "algorithmic_bytes_per_launch": alg[dom] * band_pts, "ms_per_launch": phase[dom],
                         "phases_ms": dict(zip(["forward", "backward"], phase)),
                         "note": "per-GPU figures of one band: slowest rank's phase time against the mean band size"},
            "roofline_step": {"bound": "hbm", "achieved": gbs, "peak": peak * world, "unit": "GB/s",
                              "frac": gbs / (peak * world), "peak_source": src},
            "collective": {"kind": "none (NCCL is only used for rendezvous and the timing all-reduce)" if peer is not None
                           else "NCCL send/recv (batch_isend_irecv)",
                           "data_path": transport, "halo_bytes_per_rank_per_tensor": halo_bytes,
                           "barriers_per_step": 2 if peer is not None else 0},
            "clocks": clocks, "gpu_launches": (12 + (2 if peer is not None else 0)) * args.steps}
        if e2e:
            line["e2e"] = e2e
        if batch:
            line["batch_sharded"] = batch
        print(json.dumps(line), flush=True)
    dist.destroy_process_group()
