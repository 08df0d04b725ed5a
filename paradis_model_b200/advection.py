"""Drop-in for the reference's ``model/advection.py::NeuralSemiLagrangian``.

Constructor and ``forward(hidden_features, u, v, dt)`` keep the reference's signature
(model/advection.py:10-19, 116-122), submodule names (``down_projection``, ``up_projection``,
``padding_interp``) and non-persistent buffers (58-72), so checkpoints load with
``strict=True`` and ``model/paradis.py`` runs unmodified on top of it.  Lines 129-169 of the
reference (pole mean, departure points, padding, grid_sample, pole mean) run as ONE fused
CUDA operator, ``torch.ops.paradis.sl_advect``.

Displacement limits.  The reference puts no bound on the velocities.  Here the forward accepts any displacement; the
deterministic adjoint tracks row displacements of up to 126 latitude rows (`PARADIS_SL_MAX_DISP_ROWS`).  A larger one --
or, in a latitude-band call, a departure stencil outside the band's halo -- is reported, not ignored: the kernel stores
an error code in a host-mapped status word which every later call of the operator checks on entry
(`RuntimeError: paradis_sl device status DISPLACEMENT`), and `paradis_model_b200.check_status()` checks it
synchronously.  `cfl_cells` is only a speed hint for the fused backward: planes that exceed it are recomputed by the
general path on the device.
"""
import torch

from .ops import SLGeometry, pack_tables, pack_tables64, sl_advect
from .padding import GeoCyclicPadding
from .projection import resolve_block_factory


class NeuralSemiLagrangian(torch.nn.Module):
    """Neural semi-Lagrangian advection operator (B200-native core)."""

    def __init__(self, cfg, hidden_dim: int, mesh_size: tuple, num_vels: int, lat_grid: torch.Tensor,
                 lon_grid: torch.Tensor, interpolation: str = "bicubic", math: str = "fast",
                 block_factory=None, cfl_cells: float = 8.0):
        super().__init__()
        if interpolation not in ("bilinear", "bicubic"):
            raise ValueError(f"interpolation must be 'bilinear' or 'bicubic', got {interpolation!r}")
        self.padding = 2 if interpolation == "bicubic" else 1
        self.padding_interp = GeoCyclicPadding(self.padding)  # kept for structural parity; fused in the op
        self.hidden_dim = hidden_dim
        self.num_vels = num_vels
        self.mesh_size = mesh_size
        self.interpolation = interpolation
        self.math = math
        self.cfl_cells = float(cfl_cells)  # backward performance hint, see ops.sl_advect

        block = block_factory or resolve_block_factory()
        adv_cfg = cfg.model.physblock.advection
        self.down_projection = block(layers=adv_cfg.down_projection.layers, input_dim=hidden_dim,
                                     output_dim=num_vels, mesh_size=mesh_size,
                                     hidden_dim=adv_cfg.down_projection.hidden_dim)
        self.up_projection = block(layers=adv_cfg.up_projection.layers, input_dim=num_vels,
                                   output_dim=hidden_dim, mesh_size=mesh_size,
                                   hidden_dim=adv_cfg.up_projection.hidden_dim)

        H, W = mesh_size
        if tuple(lat_grid.shape) != (H, W) or tuple(lon_grid.shape) != (H, W):
            raise ValueError("lat_grid / lon_grid must have shape mesh_size")
        if not SLGeometry.separable(lat_grid, lon_grid):
            raise ValueError("NeuralSemiLagrangian (B200) needs a separable lat-lon mesh")
        reg = lambda name, t: self.register_buffer(name, t, persistent=False)
        reg("lat_grid", lat_grid.unsqueeze(0).unsqueeze(0).contiguous().clone())
        reg("lon_grid", lon_grid.unsqueeze(0).unsqueeze(0).contiguous().clone())
        reg("Hf", torch.tensor(float(H)))
        reg("Wf", torch.tensor(float(W)))
        reg("min_lat", torch.min(lat_grid))
        reg("max_lat", torch.max(lat_grid))
        reg("min_lon", torch.min(lon_grid))
        reg("max_lon", torch.max(lon_grid))
        reg("d_lon", self.max_lon - self.min_lon)
        reg("d_lat", self.max_lat - self.min_lat)
        reg("sl_tables", torch.empty(0))
        reg("sl_tables64", torch.empty(0, dtype=torch.float64))
        self._scalars = [float(self.min_lat.float()), float(self.d_lat.float()),
                         float(self.min_lon.float()), float(self.d_lon.float())]
        # float64 inputs: the buffers as they are (the reference computes d_lat / d_lon here in the grids' dtype, and
        # .double() only converts them)
        self._scalars64 = [float(self.min_lat), float(self.d_lat), float(self.min_lon), float(self.d_lon)]
        self._refresh_tables()

    def _refresh_tables(self):
        # sin/cos of the arrival latitudes with torch's own fp32 kernels on the buffers' device,
        # exactly what the reference evaluates per call (advection.py:86-87)
        lat = self.lat_grid[0, 0, :, 0].float()
        lon = self.lon_grid[0, 0, 0, :].float()
        self.sl_tables = pack_tables(lat, lon)
        # float64 inputs: the same with torch's fp64 kernels from the grids' own values (the reference after .double())
        self.sl_tables64 = pack_tables64(self.lat_grid[0, 0, :, 0], self.lon_grid[0, 0, 0, :])

    def _apply(self, fn, *args, **kwargs):
        out = super()._apply(fn, *args, **kwargs)
        self._refresh_tables()
        return out

    def geometry(self) -> SLGeometry:
        H, W = self.mesh_size
        return SLGeometry(self.sl_tables, self._scalars, H, W, tables64=self.sl_tables64, scalars64=self._scalars64)

    def forward(self, hidden_features: torch.Tensor, u: torch.Tensor, v: torch.Tensor, dt: float) -> torch.Tensor:
        """Compute advection using rotated coordinate system."""
        projected = self.down_projection(hidden_features)
        advected = sl_advect(projected, u, v, self.geometry(), dt, self.interpolation, True, self.math,
                             self.cfl_cells)
        return self.up_projection(advected)
