"""Native bf16 storage of the GeoCyclic ops (include/paradis_geocyclic.h, ops.NATIVE_BF16): with bf16 activations the
pad, depthwise-convolution and avgpool5 kernels read and write bf16.  Every comparison is torch.equal against the upcast
path -- the fp32 kernels on .float() copies, results cast back by .to(torch.bfloat16) -- and, for the avgpool5 adjoint,
against the full-resolution composition it replaces."""
import pytest
import torch

from paradis_model_b200 import blocks, ops

pytestmark = pytest.mark.gpu
BF = torch.bfloat16


@pytest.fixture(autouse=True)
def _restore_switches():
    yield
    ops.NATIVE_BF16 = True


def _randn(shape, seed, dtype=BF):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(shape, generator=g).cuda().to(dtype)


# ----------------------------------------------------------------------------------------------------------------------
# pad
# ----------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("p", [1, 2, 3])
@pytest.mark.parametrize("shape", [(2, 3, 6, 8), (2, 3, 33, 64), (1, 2, 721, 1440)])
def test_pad_forward_backward(shape, p):
    B, Cn, H, W = shape
    x = _randn(shape, 10 * p + H)
    gy = _randn((B, Cn, H + 2 * p, W + 2 * p), 10 * p + H + 1)
    xc = x.clone().requires_grad_(True)
    y = ops.geocyclic_pad(xc, p)
    y.backward(gy)
    y_ref = torch.ops.paradis.geocyclic_pad(x.float(), p).to(BF)
    gx_ref = torch.ops.paradis.geocyclic_pad_backward(gy.float(), p).to(BF)
    assert y.dtype == BF and torch.equal(y, y_ref)
    assert xc.grad.dtype == BF and torch.equal(xc.grad, gx_ref)


# ----------------------------------------------------------------------------------------------------------------------
# dwconv
# ----------------------------------------------------------------------------------------------------------------------
def _dw_inputs(shape, k, seed):
    B, Cn, H, W = shape
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, Cn, H, W, generator=g).cuda().to(BF)
    w = (torch.randn(Cn, 1, k, k, generator=g) / k).cuda()
    b = torch.randn(Cn, generator=g).cuda()
    gy = torch.randn(B, Cn, H, W, generator=g).cuda().to(BF)
    return x, w, b, gy


def _dw_run(x, w, b, gy, req=(True, True, True)):
    xc, wc = x.clone().requires_grad_(req[0]), w.clone().requires_grad_(req[1])
    bc = b.clone().requires_grad_(req[2]) if b is not None else None
    y = ops.geocyclic_dwconv(xc, wc, bc)
    y.backward(gy)
    return y.detach(), xc.grad, wc.grad, (bc.grad if bc is not None else None)


def _dw_check(x, w, b, gy, req=(True, True, True)):
    got = _dw_run(x, w, b, gy, req)
    ref = _dw_run(x.float(), w, b, gy.float(), req)
    assert got[0].dtype == BF and torch.equal(got[0], ref[0].to(BF)), "y"
    if req[0]:
        assert got[1].dtype == BF and torch.equal(got[1], ref[1].to(BF)), "grad input"
    else:
        assert got[1] is None
    for k, name in ((2, "grad weight"), (3, "grad bias")):
        if ref[k] is None:
            assert got[k] is None, name
        else:
            assert got[k].dtype == torch.float32 and torch.equal(got[k], ref[k]), name
    return got


@pytest.mark.parametrize("bias", [True, False])
@pytest.mark.parametrize("k", [3, 5, 7])
@pytest.mark.parametrize("shape", [(2, 5, 33, 64), (1, 3, 128, 256), (1, 2, 721, 1440), (3, 4, 9, 38)])
def test_dwconv_forward_backward(shape, k, bias):
    x, w, b, gy = _dw_inputs(shape, k, k * 100 + shape[2])
    b = b if bias else None
    first = _dw_check(x, w, b, gy)
    again = _dw_run(x, w, b, gy)
    for a, c in zip(first, again):
        assert (a is None and c is None) or torch.equal(a, c)


@pytest.mark.parametrize("req", [(True, False, False), (False, True, True)], ids=["input-only", "weight-only"])
@pytest.mark.parametrize("k", [3, 7])
def test_dwconv_partial_requires_grad(req, k):
    x, w, b, gy = _dw_inputs((2, 5, 33, 64), k, 7 + k)
    _dw_check(x, w, b, gy, req)


# ----------------------------------------------------------------------------------------------------------------------
# avgpool5
# ----------------------------------------------------------------------------------------------------------------------
def _composition(gy32, shape, s):
    """The adjoint as it was built before it had a kernel of its own: grad_y scattered into a zero-filled
    full-resolution grid, then the depthwise grad-input kernels with the 1/25 box filter."""
    B, Cn, H, W = shape
    g_full = torch.zeros(shape, dtype=torch.float32, device=gy32.device)
    g_full[:, :, ::s, ::s] = gy32
    box = torch.full((Cn, 1, 5, 5), 1.0 / 25.0, dtype=torch.float32, device=gy32.device)
    gx, _, _ = torch.ops.paradis.geocyclic_dwconv_backward(g_full, g_full, box, True, False, False)
    return gx


POOL_SHAPES = [(2, 3, 35, 62), (1, 2, 30, 50), (1, 2, 721, 1440)]


@pytest.mark.parametrize("stride", [1, 2, 3, 4])
@pytest.mark.parametrize("shape", POOL_SHAPES)
def test_avgpool5_fp32_adjoint_equals_composition(shape, stride):
    B, Cn, H, W = shape
    x = _randn(shape, stride, torch.float32)
    gy = _randn((B, Cn, (H - 1) // stride + 1, (W - 1) // stride + 1), stride + 1, torch.float32)
    gy[:, :, ::3, ::2] = 0.0                              # exact zeros of both signs among the non-zero terms
    gy[:, :, 1::3, ::2] = -0.0
    xc = x.clone().requires_grad_(True)
    ops.geocyclic_avgpool5(xc, stride).backward(gy)
    ref = _composition(gy, shape, stride)
    assert xc.grad.dtype == torch.float32 and torch.equal(xc.grad, ref)
    assert torch.equal(torch.ops.paradis.geocyclic_avgpool5_backward(gy, H, W, stride), ref)


@pytest.mark.parametrize("stride", [1, 2, 3, 4])
@pytest.mark.parametrize("shape", POOL_SHAPES)
def test_avgpool5_bf16_forward_backward(shape, stride):
    B, Cn, H, W = shape
    x = _randn(shape, 20 + stride)
    gy = _randn((B, Cn, (H - 1) // stride + 1, (W - 1) // stride + 1), 21 + stride)
    xc = x.clone().requires_grad_(True)
    y = ops.geocyclic_avgpool5(xc, stride)
    y.backward(gy)
    assert y.dtype == BF and torch.equal(y, torch.ops.paradis.geocyclic_avgpool5(x.float(), stride).to(BF))
    assert xc.grad.dtype == BF and torch.equal(xc.grad, _composition(gy.float(), shape, stride).to(BF))


# ----------------------------------------------------------------------------------------------------------------------
# no casts, less memory, ineligible calls
# ----------------------------------------------------------------------------------------------------------------------
def _step(op, x, w, b, gy):
    xc = x.clone().requires_grad_(True)
    if op == "pad":
        y = ops.geocyclic_pad(xc, 2)
    elif op == "dwconv":
        y = ops.geocyclic_dwconv(xc, w, b)
    else:
        y = ops.geocyclic_avgpool5(xc, 2)
    y.backward(gy)
    return y.detach(), xc.grad


def _step_inputs(op, shape, dtype=BF, seed=0):
    B, Cn, H, W = shape
    x = _randn(shape, seed, dtype)
    w = (0.2 * _randn((Cn, 1, 5, 5), seed + 1, torch.float32)).requires_grad_(True)
    b = _randn((Cn,), seed + 2, torch.float32).requires_grad_(True)
    out = {"pad": (H + 4, W + 4), "dwconv": (H, W), "avgpool5": ((H - 1) // 2 + 1, (W - 1) // 2 + 1)}[op]
    gy = _randn((B, Cn) + out, seed + 3, dtype)
    return x, w, b, gy


def _ops_in(fn):
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return {e.name for e in prof.events()}


@pytest.mark.parametrize("op", ["pad", "dwconv", "avgpool5"])
def test_native_call_launches_no_cast(op):
    x, w, b, gy = _step_inputs(op, (2, 4, 64, 128))
    step = lambda: _step(op, x, w, b, gy)
    step()                                                   # warm-up (library load)
    names = _ops_in(step)
    assert "aten::_to_copy" not in names, sorted(names)
    ops.NATIVE_BF16 = False
    assert "aten::_to_copy" in _ops_in(step)


def _peak(op, x, w, b, gy):
    _step(op, x, w, b, gy)                                   # warm-up: allocator pools, library
    w.grad = b.grad = None
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    _step(op, x, w, b, gy)
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    w.grad = b.grad = None
    return peak


@pytest.mark.parametrize("op", ["pad", "dwconv"])
def test_peak_memory_lower_than_upcast(op):
    x, w, b, gy = _step_inputs(op, (1, 64, 181, 360), seed=4)
    native = _peak(op, x, w, b, gy)
    ops.NATIVE_BF16 = False
    upcast = _peak(op, x, w, b, gy)
    one_copy = x.numel() * 4
    assert upcast - native >= one_copy, (native, upcast, one_copy)


@pytest.mark.parametrize("dtype", [torch.float16, torch.float32])
@pytest.mark.parametrize("op", ["pad", "dwconv", "avgpool5"])
def test_ineligible_calls_unchanged(op, dtype):
    x, w, b, gy = _step_inputs(op, (2, 3, 33, 64), dtype, seed=5)
    runs = []
    for native in (True, False):
        ops.NATIVE_BF16 = native
        runs.append(_step(op, x, w, b, gy))
    for a, c in zip(*runs):
        assert a.dtype == dtype and c.dtype == dtype and torch.equal(a, c)


# ----------------------------------------------------------------------------------------------------------------------
# compile / autocast / checkpoint, the blocks, the whole model
# ----------------------------------------------------------------------------------------------------------------------
def test_compile_autocast_checkpoint_bit_equal_to_eager():
    from torch.utils.checkpoint import checkpoint
    x = _randn((2, 4, 32, 64), 30)
    w = 0.2 * _randn((4, 1, 3, 3), 31, torch.float32)
    b = _randn((4,), 32, torch.float32)

    def fn(a, wc, bc):
        y = ops.geocyclic_pad(a, 1)                          # [2, 4, 34, 66]
        y = ops.geocyclic_dwconv(y, wc, bc)
        return ops.geocyclic_avgpool5(y, 2)

    gy = _randn((2, 4, 17, 33), 33)

    def grads(call, amp=False, ckpt=False):
        a, wc, bc = x.clone().requires_grad_(True), w.clone().requires_grad_(True), b.clone().requires_grad_(True)
        with torch.autocast("cuda", dtype=BF, enabled=amp):
            out = checkpoint(call, a, wc, bc, use_reentrant=False) if ckpt else call(a, wc, bc)
        out.backward(gy)
        return out.detach(), a.grad, wc.grad, bc.grad

    eager = grads(fn)
    assert eager[0].dtype == BF and eager[1].dtype == BF and eager[2].dtype == torch.float32
    compiled = torch.compile(fn, fullgraph=True)
    for other in (grads(compiled), grads(fn, amp=True), grads(fn, ckpt=True), grads(compiled, amp=True)):
        for a, c in zip(eager, other):
            assert a.dtype == c.dtype and torch.equal(a, c)


@pytest.fixture
def _deterministic_cudnn():
    old = torch.backends.cudnn.deterministic
    torch.backends.cudnn.deterministic = True
    yield
    torch.backends.cudnn.deterministic = old


def _module_step(m, x, gy):
    m.zero_grad(set_to_none=True)
    xc = x.clone().requires_grad_(True)
    with torch.autocast("cuda", dtype=BF):
        y = m(xc)
    y.backward(gy)
    return [y.detach(), xc.grad] + [p.grad.clone() for p in m.parameters()]


@pytest.mark.usefixtures("_deterministic_cudnn")
@pytest.mark.parametrize("kind", ["SepConv3", "SepConv5", "SepConv7", "Downsample2", "Downsample4"])
def test_blocks_bit_equal_to_upcast(kind):
    torch.manual_seed(0)
    k = int(kind[-1])
    m = (blocks.SepConv(6, 8, (33, 64), kernel_size=k) if kind.startswith("Sep") else
         blocks.PhysicalDownsample(stride=k)).cuda()
    x = _randn((2, 6, 33, 64), 40 + k)
    out_shape = (2, 8, 33, 64) if kind.startswith("Sep") else (2, 6, (33 - 1) // k + 1, (64 - 1) // k + 1)
    gy = _randn(out_shape, 50 + k)
    runs = []
    for native in (True, False, False):
        ops.NATIVE_BF16 = native
        runs.append(_module_step(m, x, gy))
    assert runs[0][0].dtype == BF and runs[0][1].dtype == BF
    for a, c in zip(runs[1], runs[2]):                        # control: the upcast arm is reproducible
        assert torch.equal(a, c)
    for a, c in zip(runs[0], runs[1]):
        assert a.dtype == c.dtype and torch.equal(a, c)


@pytest.mark.usefixtures("_deterministic_cudnn")
def test_whole_model_autocast_bit_equal_to_upcast():
    """Assembly(dropin=True) from default_cfg() (latent 16, 8 velocity vectors, 2 layers, bicubic) at 64 x 128: one eager
    fwd + bwd under bf16 autocast, loss and every parameter gradient, native against upcast."""
    from oracle import paradis_assembly as A
    from oracle.sl_oracle import make_grids
    import paradis_model_b200 as P
    H, W = 64, 128
    lat, lon = make_grids(H, W, True)
    torch.manual_seed(0)
    model = A.Assembly(A.FakeDataModule, A.default_cfg(), lat, lon, dropin=True).cuda()
    g = torch.Generator().manual_seed(6)
    x = torch.randn(2, 22, H, W, generator=g).cuda()
    tgt = torch.randn(2, 7, H, W, generator=g).cuda()

    def step(native):
        ops.NATIVE_BF16 = native
        model.zero_grad(set_to_none=True)
        with torch.autocast("cuda", dtype=BF):
            loss = torch.nn.functional.mse_loss(model(x).float(), tgt)
        loss.backward()
        P.check_status()
        return [loss.detach()] + [p.grad.clone() if p.grad is not None else None for p in model.parameters()]

    up1, up2 = step(False), step(False)
    for a, c in zip(up1, up2):                                # control: cuDNN and the rest are reproducible
        assert (a is None and c is None) or torch.equal(a, c), "upcast arm not reproducible"
    nat = step(True)
    names = ["loss"] + [n for n, _ in model.named_parameters()]
    for n, a, c in zip(names, nat, up1):
        assert (a is None and c is None) or (a.dtype == c.dtype and torch.equal(a, c)), n
