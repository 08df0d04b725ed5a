"""CPU tests of the boundary: the library builds/loads, exports every symbol the header
declares, and rejects bad arguments with the documented codes before touching a GPU; bench.py's output line and
output dumps (the b200 arm's on the GPU)."""
import ctypes as C
import os
import re

import pytest

from conftest import ROOT
from paradis_model_b200 import _lib, build


def header_functions():
    text = open(os.path.join(ROOT, "include", "paradis_sl.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(paradis_[a-z0-9_]+)\s*\(", text)))


def test_library_builds_and_loads():
    path = build.build_library()
    assert os.path.exists(path)
    assert _lib.lib().paradis_sl_abi_version() == 2


def test_exports_every_declared_symbol():
    names = header_functions()
    assert len(names) == 17
    handle = C.CDLL(build.build_library())
    for n in names:
        assert hasattr(handle, n), f"{n} declared in include/paradis_sl.h but not exported"
    assert sorted(_lib.exported_symbols()) == names  # ctypes prototypes cover the whole header


def test_geom_struct_layout_matches_header():
    # 2 x int32, 3 pointers, 4 floats, 6 x int32, 2 pointers, int32
    assert C.sizeof(_lib.Geom) == 8 + 24 + 16 + 24 + 16 + 8 + 48 + 8   # + field peers, + 6 arrival peers, int32s + padding


def test_argument_errors_without_gpu():
    L = _lib.lib()
    g = _lib.Geom()
    g.H, g.W = 8, 9
    g.sin_lat = g.cos_lat = g.lon = 1  # non-NULL dummies, never dereferenced on the host
    g.own_rows = g.arr_rows = g.fld_rows = 8
    one = C.c_void_p(16)
    rc = L.paradis_sl_advect_fwd(C.byref(g), one, one, one, one, 1, 1, 72, 72, 72, 0.1, 1, 1, 0, None, 0, None, None)
    assert rc == 2 and b"even" in L.paradis_last_error()          # model/padding.py:21
    g.W = 8
    rc = L.paradis_sl_advect_fwd(C.byref(g), one, one, one, one, 1, 1, 64, 64, 64, 0.1, 3, 1, 0, None, 0, None, None)
    assert rc == 3
    rc = L.paradis_sl_advect_fwd(C.byref(g), None, one, one, one, 1, 1, 64, 64, 64, 0.1, 1, 1, 0, None, 0, None, None)
    assert rc == 4
    rc = L.paradis_sl_advect_fwd(C.byref(g), one, one, one, one, 1, 1, 64, 64, 64, 0.1, 1, 1, 0, None, 0, None, None)
    assert rc == 5  # pole_fix needs the workspace
    g.own_rows = 9
    rc = L.paradis_sl_advect_fwd(C.byref(g), one, one, one, one, 1, 1, 64, 64, 64, 0.1, 1, 0, 0, None, 0, None, None)
    assert rc == 1
    assert L.paradis_geocyclic_pad_fwd(one, one, 1, 4, 7, 1, None) == 2
    assert L.paradis_geocyclic_pad_fwd(None, one, 1, 4, 8, 1, None) == 4
    assert L.paradis_sl_advect_bwd_workspace(1, 64, 721, 1440) > 64 * 721 * 1440
    assert L.paradis_sl_host_scratch_bytes(32, 64, 4) > 8 * 4 * 32 * 64 * 4


def test_ops_fail_loudly_on_cpu():
    import torch
    import paradis_model_b200 as P
    lat, lon = __import__("oracle.sl_oracle", fromlist=["x"]).make_grids(8, 16, True)
    geo = P.SLGeometry.from_grids(lat, lon)
    x = torch.zeros(1, 1, 8, 16)
    with pytest.raises((RuntimeError, NotImplementedError)):
        P.sl_advect(x, x, x, geo, 0.1)
    with pytest.raises((RuntimeError, NotImplementedError)):
        P.geocyclic_pad(x, 1)


def test_bench_reference_arm_prints_the_contract_line(tmp_path):
    """`bench.py --impl reference` (the CPU arm run beside the GPU arm) needs no GPU: one JSON line
    with the same metric / unit / config as the product arm plus impl, cpu_baseline and a zero-copy e2e object;
    --dump-outputs writes the four arrays of the last timed step."""
    import json, os, subprocess, sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    res = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "0", "--workload", "c2", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=600, cwd=root)
    assert res.returncode == 0, res.stderr[-2000:]
    line = json.loads(res.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "grid-pt*ch/s" and line["higher_is_better"] is True
    assert line["metric"] == "SL advection fwd+bwd grid-pts*ch/s" and line["value"] > 0
    assert line["cpu_baseline"]["kind"] in ("port", "reference") and line["cpu_baseline"]["cores"] >= 1
    assert line["cpu_baseline"]["value"] == line["value"] and line["cpu_baseline"]["sample"]
    assert line["e2e"] == {"value": line["value"], "unit": line["unit"], "h2d_bytes_per_step": 0,
                           "d2h_bytes_per_step": 0}
    assert "workload" in line["config"] and line["n_gpus"] == 1 and line["vs_baseline"] is None
    # c2 mesh (128 x 256, no pole rows), the 8-channel CPU sample, seed 0: small enough to be written whole
    import numpy as np
    import torch
    from conftest import relmax
    from oracle import sl_oracle as O
    from paradis_model_b200 import synthetic as S
    field, u, v, go = S.white_noise_inputs(128, 256, 1, 8)
    lat, lon = O.make_grids(128, 256, False)
    ref = O.sl_advect_fwd_bwd(field, u, v, lat, lon, S.DT_DEFAULT, go, "bilinear")
    assert sorted(os.listdir(tmp_path)) == ["grad_field.npy", "grad_u.npy", "grad_v.npy", "out.npy"]
    for name, r in zip(("out", "grad_field", "grad_u", "grad_v"), ref):
        a = np.load(tmp_path / f"{name}.npy")
        assert a.dtype == np.float32 and a.shape == tuple(r.shape), name
        assert relmax(torch.from_numpy(a), r) < 1e-5, name


@pytest.mark.gpu
def test_bench_b200_arm_dumps_a_sample_of_the_last_step(tmp_path):
    """`bench.py --dump-outputs` on c2 ([8, 64, 128, 256]: more elements than DUMP_SAMPLES): four float32 files holding
    the timed path's outputs at sample_index(numel), bit for bit what RawAdvection computes from the same seeded inputs
    in this process, and within the white-noise tolerances of the oracle run by torch on the same GPU."""
    import importlib.util, subprocess, sys
    import numpy as np
    import torch
    import paradis_model_b200 as P
    from conftest import bad_fraction
    from oracle import sl_oracle as O
    from paradis_model_b200 import synthetic as S
    from paradis_model_b200.ops import RawAdvection
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1", "--workload",
                          "c2", "--no-cpu", "--no-e2e", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert res.returncode == 0, res.stderr[-2000:]
    spec = importlib.util.spec_from_file_location("bench", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    H, W, V, B, poles = bench.WORKLOADS["c2"]
    idx = torch.from_numpy(bench.sample_index(B * V * H * W)).cuda()
    assert 0 < idx.numel() <= bench.DUMP_SAMPLES < B * V * H * W
    field, u, v, go = [t.cuda() for t in S.white_noise_inputs(H, W, B, V)]
    lat, lon = [t.cuda() for t in S.make_grids(H, W, poles)]
    R = RawAdvection(P.SLGeometry.from_grids(lat, lon), B, V, "bilinear", True, "fast", bench.CFL_CELLS)
    R.forward(field, u, v, S.DT_DEFAULT)
    R.backward(go, field, u, v, S.DT_DEFAULT, 3)
    P.check_status()
    ref = O.sl_advect_fwd_bwd(field, u, v, lat, lon, S.DT_DEFAULT, go, "bilinear")
    assert sorted(os.listdir(tmp_path)) == ["grad_field.npy", "grad_u.npy", "grad_v.npy", "out.npy"]
    for k, (name, mine) in enumerate(zip(bench.OUTPUT_NAMES, (R.out, R.gfield, R.gu, R.gv))):
        a = np.load(tmp_path / f"{name}.npy")
        assert a.dtype == np.float32 and a.shape == tuple(idx.shape), name
        a = torch.from_numpy(a)
        assert torch.equal(a, mine.reshape(-1)[idx].cpu()), name
        if k < 3:      # the tolerances of test_fast_mode_white_noise_statistics
            assert bad_fraction(a, ref[k].reshape(-1)[idx].cpu(), 1e-3 if k == 2 else 1e-4) < (2e-3 if k == 2 else 1e-3), name
