"""The boundary kernels of ops.cu against float64 (or exact) references: BGNet's instance-norm apply (+ReLU, +residual) and
the statistics it uses, the tanh head of BGNet, the NCHW <-> planes layout converters with channel windows, and the
uint8 frame conversion every output frame passes through."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from test_attention_gpu import SENTINEL16, _raw_planes, check_outside_kept, format_unit

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
GRID_STRIDE = 148 * 16 * 256      # elements one launch of the element-wise kernels covers before striding


def _rand(shape, seed, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    return (torch.rand(shape, generator=g) * 2 - 1) * scale


def _sentinel_planes(P, N, H, W, C, pitch, coff):
    from ipercore_b200.ops import Planes
    buf = Planes.empty(P, N, H, W, C, DEV, pitch=pitch)
    buf.data.view(torch.int16).fill_(SENTINEL16)
    return buf, buf.window(coff, C), [t.clone() for t in _raw_planes(buf)]


def _planes_window(x, P, pitch, coff, seed):
    """x (N,C,H,W) stored as channels [coff, coff+C) of a planes buffer whose other channels hold other values"""
    from ipercore_b200.ops import Planes
    N, C, H, W = x.shape
    wide = torch.cat([_rand((N, coff, H, W), seed), x, _rand((N, pitch - coff - C, H, W), seed + 1)], 1)
    return Planes.from_nchw(wide.to(DEV), P).window(coff, C)


# ----------------------------------------------------------------------------------------------------------------------
# instance norm
# ----------------------------------------------------------------------------------------------------------------------
def _instnorm_apply_case(N, H, W, windows, relu, residual, P):
    from ipercore_b200 import ops
    C = 64
    xv = _rand((N, C, H, W), 81, 2.0) + _rand((1, C, 1, 1), 82, 1.5)
    x = _planes_window(xv, P, 96, 16, 83) if windows else _planes_window(xv, P, C, 0, 83)
    res = None
    if residual:
        res = _planes_window(_rand((N, C, H, W), 84), P, 80, 8, 85) if windows else _planes_window(_rand((N, C, H, W), 84), P, C, 0, 85)
    pitch, coff = (88, 24) if windows else (C, 0)
    buf, out, before = _sentinel_planes(P, N, H, W, C, pitch, coff)
    stats = ops.instnorm_stats(x)
    ops.instnorm_apply(x, stats, out, relu=relu, res=res)
    torch.cuda.synchronize()
    xs = x.to_nchw().cpu().double()
    exp = F.instance_norm(xs, eps=1e-5)
    if relu:
        exp = exp.clamp_min(0)
    if residual:
        exp = exp + res.to_nchw().cpu().double()
    from ipercore_b200.ops import Planes
    exp_r = Planes.from_nchw(exp.float().to(DEV), P).to_nchw()
    got = out.to_nchw()
    assert torch.isfinite(got).all()
    err = (got - exp_r).abs()
    # fp32 normalisation of values up to ~4 sigma (fp32 mean / rstd, one subtract, one multiply, one add): 1e-6
    tol = 1e-6 + format_unit(exp_r.abs(), P)
    print("instnorm_apply N=%d %dx%d relu=%d res=%d P=%d: max |err| %.2e (%.2f of the bound)"
          % (N, H, W, relu, residual, P, float(err.max()), float((err / tol).max())))
    assert (err <= tol).all()
    check_outside_kept(buf, before, coff, C, "instnorm_apply")


@pytest.mark.parametrize("P", [1, 2, 3])
@pytest.mark.parametrize("residual", [False, True])
@pytest.mark.parametrize("relu", [False, True])
def test_instnorm_apply(relu, residual, P):
    """out = [res +] [relu](IN(x)) (bg_inpaintor.py:13-21, 33-52) with x, res and out as channel windows"""
    _instnorm_apply_case(2, 13, 11, True, relu, residual, P)


def test_instnorm_apply_large():
    """2 x 96 x 96 x 64 elements: more than one grid-stride trip, in BGNet's residual form"""
    assert 2 * 96 * 96 * 64 > GRID_STRIDE
    _instnorm_apply_case(2, 96, 96, False, True, True, 2)


def test_instnorm_stats_fp64():
    """mean / rstd of the stored values against float64, with one channel whose offset dominates its spread (mean 50,
    std 0.05): there E[x^2] - mean^2 cancels 6 digits, which is what the fp32-partial / fp64-fold scheme has to carry."""
    from ipercore_b200 import ops
    N, C, H, W = 2, 64, 256, 256
    g = torch.Generator().manual_seed(91)
    xv = torch.randn((N, C, H, W), generator=g) * (torch.rand((1, C, 1, 1), generator=g) * 2 + 0.1) \
        + (torch.rand((1, C, 1, 1), generator=g) * 4 - 2)
    xv[1, 5] = 50.0 + 0.05 * torch.randn((H, W), generator=g)
    x = _planes_window(xv, 2, 80, 8, 92)
    stats = ops.instnorm_stats(x).cpu().double()
    xs = x.to_nchw().cpu().double()
    mean = xs.mean((2, 3))
    rstd = 1.0 / torch.sqrt(xs.var((2, 3), unbiased=False) + 1e-5)
    em = (stats[..., 0] - mean).abs()
    er = ((stats[..., 1] - rstd) / rstd).abs()
    em[1, 5] = er[1, 5] = 0
    om, orr = abs(float(stats[1, 5, 0] - mean[1, 5])), abs(float((stats[1, 5, 1] - rstd[1, 5]) / rstd[1, 5]))
    print("instnorm_stats: max |mean err| %.2e, max rstd rel err %.2e; offset channel (mean 50, std 0.05): "
          "|mean err| %.2e, rstd rel err %.2e" % (float(em.max()), float(er.max()), om, orr))
    assert float(em.max()) <= 1e-6 and float(er.max()) <= 2e-6
    # one fp32 step of 50 is 3.8e-6; the rstd bound is provisional, to be set from the measured value
    assert om <= 4e-6 and orr <= 2e-3


# ----------------------------------------------------------------------------------------------------------------------
# tanh head, layout converters
# ----------------------------------------------------------------------------------------------------------------------
def _ulp32(a):
    e = torch.frexp(a.abs().float().clamp_min(2.0 ** -126)).exponent
    return torch.ldexp(torch.ones_like(a, dtype=torch.float64), e - 24)


@pytest.mark.parametrize("pitch", [3, 8])
def test_tanh_nhwc_to_nchw(pitch):
    """BGNet's last layer: tanh of the first 3 channels of an NHWC fp32 map (pitch 3 is BGNet's own call), within 2 fp32 ulp"""
    from ipercore_b200 import ops
    N, H, W, C = 2, 7, 9, 3
    x = _rand((N, H, W, pitch), 101, 4.0)
    x.view(-1)[:8] = torch.tensor([0.0, -0.0, 1e-8, -1e-8, 9.0, -9.0, 20.0, -20.0])
    got = ops.tanh_nhwc_to_nchw(x.to(DEV), C).cpu().double()
    exp = torch.tanh(x[..., :C].double()).permute(0, 3, 1, 2)
    ulps = ((got - exp).abs() / _ulp32(exp)).max()
    print("tanh pitch %d: max error %.2f fp32 ulp" % (pitch, float(ulps)))
    assert float(ulps) <= 2.0


@pytest.mark.parametrize("P", [1, 2, 3])
@pytest.mark.parametrize("N,C,pitch,coff", [(2, 4, 8, 4), (3, 192, 208, 8), (2, 64, 64, 0)])
def test_nchw_planes_round_trip(N, C, pitch, coff, P):
    """nchw_to_planes into a window of a sentinel buffer, planes_to_nchw back; 7 x 9 pixels (not a multiple of the 32-pixel
    transpose tile), C not a multiple of 32"""
    from ipercore_b200.ops import Planes
    H, W = 7, 9
    x = _rand((N, C, H, W), 111)
    if P == 1:
        x = x.half().float()        # fp16-representable: the single plane holds it exactly
    buf, win, before = _sentinel_planes(P, N, H, W, C, pitch, coff)
    Planes.from_nchw(x.to(DEV), P, out=win)
    back = win.to_nchw().cpu()
    check_outside_kept(buf, before, coff, C, "nchw_to_planes")
    err = (back.double() - x.double()).abs()
    # P=2: hi + lo keeps 22 bits (2^-21 relative) down to the lo plane's subnormal step; P=3: the e4m3 remainder, 15 bits
    bound = {1: 0 * x.abs(), 2: x.abs() * 2.0 ** -21 + 2.0 ** -25, 3: x.abs() * 2.0 ** -15 + 2.0 ** -23}[P].double()
    print("planes round trip N=%d C=%d window %d/%d P=%d: max |err| %.2e" % (N, C, coff, pitch, P, float(err.max())))
    assert (err <= bound).all()


@pytest.mark.parametrize("N,C,pitch,coff", [(2, 4, 8, 4), (3, 192, 208, 8), (2, 3, 8, 5)])
def test_nhwc_f32_to_nchw_window(N, C, pitch, coff):
    """iper_nhwc_f32_to_nchw with a channel window (the wrapper always passes pitch = C, coff = 0): a bit-exact copy"""
    from ipercore_b200 import _lib, ops
    H, W = 7, 9
    x = _rand((N, H, W, pitch), 121).to(DEV)
    out = torch.empty((N, C, H, W), dtype=torch.float32, device=DEV)
    out.view(torch.int32).fill_(0x7FC0DEAD)
    _lib.check(_lib.lib.iper_nhwc_f32_to_nchw(x.data_ptr(), N, C, H * W, pitch, coff, out.data_ptr(), ops._stream()),
               "nhwc_f32_to_nchw")
    exp = x[..., coff:coff + C].permute(0, 3, 1, 2)
    assert torch.equal(out.view(torch.int32), exp.contiguous().view(torch.int32))
    full = ops.nhwc_f32_to_nchw(x)
    assert torch.equal(full.view(torch.int32), x.permute(0, 3, 1, 2).contiguous().view(torch.int32))


# ----------------------------------------------------------------------------------------------------------------------
# uint8 frames
# ----------------------------------------------------------------------------------------------------------------------
def _u8_expected(pred):
    """cv_utils.save_cv2_img: (x + 1) / 2.0 * 255 in float32, astype(np.uint8), RGB -> BGR; pred (B,3,S,S) -> (B,S,S,3).
    Inside [-1, 1] the clip is a no-op and this is exactly the reference's conversion; outside, numpy's float -> uint8
    cast is undefined and the kernel clamps to 0 / 255 (its choice, modelled by the clip)."""
    r = (pred + 1) / 2.0 * 255
    assert r.dtype == np.float32
    inside = (pred >= -1) & (pred <= 1)
    assert (r[inside] >= 0).all() and (r[inside] < 256).all()
    return np.clip(r, 0, 255).astype(np.uint8).transpose(0, 2, 3, 1)[..., ::-1]


def test_pred_to_u8_boundaries():
    """every code boundary k/127.5 - 1 and both fp32 neighbours (truncation, not rounding), +-1, values just outside"""
    from ipercore_b200 import ops
    k = (np.arange(256, dtype=np.float32) / np.float32(127.5) - 1).astype(np.float32)
    vals = np.concatenate([k, np.nextafter(k, np.float32(2)), np.nextafter(k, np.float32(-2)),
                           np.array([-1, 1, -1 - 2 ** -23, 1 + 2 ** -23, -1.01, 1.01, -3, 3], np.float32)])
    S = 32
    g = np.random.default_rng(131)
    pred = np.stack([np.resize(vals[g.permutation(len(vals))], (S, S)) for _ in range(3)])[None].astype(np.float32)
    got = ops.pred_to_u8(torch.from_numpy(pred).to(DEV)).cpu().numpy()
    exp = _u8_expected(pred)
    assert np.array_equal(got, exp), "%d codes differ" % int((got != exp).sum())
    assert got[pred.transpose(0, 2, 3, 1)[..., ::-1] < -1].max() == 0 and got[pred.transpose(0, 2, 3, 1)[..., ::-1] > 1].min() == 255


def test_pred_to_u8_large():
    """B*S*S above one grid-stride trip"""
    from ipercore_b200 import ops
    B, S = 3, 512
    assert B * S * S > GRID_STRIDE
    pred = (_rand((B, 3, S, S), 141) * 1.02).numpy()
    got = ops.pred_to_u8(torch.from_numpy(pred).to(DEV)).cpu().numpy()
    assert np.array_equal(got, _u8_expected(pred))
