"""GPU parity of the tcgen05 implicit-GEMM convolution: against a plain PyTorch fp32 convolution (CPU) of the same
operands and against the CUDA-core cross-check kernel, for every mode / epilogue / tile width the generator uses."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

DEV = "cuda:0"


def _rand(shape, seed, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    return (torch.rand(shape, generator=g) * 2 - 1) * scale


def _planes_value(p):
    return p.to_nchw().cpu()


def _ref_conv(x, w, mode, k):
    if mode == 0:
        return F.conv2d(x, w, padding=k // 2)
    if mode == 1:
        return F.conv2d(x, w, stride=2, padding=1)
    return F.conv_transpose2d(x, w, stride=2, padding=1)


# (N, H, W, Cin, Cout, mode, k): shapes cover block_n 64/128/256, multi n-tile (512 rows), partial tiles, tn>1
CASES = [
    (2, 16, 16, 64, 64, 0, 3), (1, 32, 32, 128, 128, 0, 3), (2, 16, 16, 256, 256, 0, 3), (3, 8, 8, 64, 256, 0, 1),
    (1, 20, 12, 64, 64, 0, 3), (2, 32, 32, 64, 128, 1, 3), (2, 16, 16, 128, 256, 1, 3),
    (2, 8, 8, 256, 256, 2, 4), (1, 16, 16, 256, 128, 2, 4), (1, 16, 16, 128, 64, 2, 4), (1, 16, 16, 384, 256, 0, 3),
    # halo kernel (cta_pair=2): partial 16x8 tiles, an odd tile count (the pair's second tile is empty), two n tiles
    (1, 20, 24, 64, 128, 0, 3), (3, 8, 16, 128, 128, 0, 3), (1, 24, 40, 128, 512, 0, 3), (3, 8, 16, 128, 64, 2, 4),
]


def _halo_ok(mode, k, bn, H, W):
    """layers the vertical-halo CTA-pair kernel accepts (iper_conv_gemm, cta_pair = 2)"""
    return H >= 8 and W >= 16 and ((mode == 0 and k == 3 and bn >= 64) or (mode == 2 and bn == 64))


def _operand_terms(x, P):
    """(x_main, x_lo_term, x_a8_term) exactly as the three MMA groups of format P see the activation."""
    from ipercore_b200 import ops
    hi = x.half().float()
    if P == 1:
        return hi, None, None
    if P == 2:
        return hi, (x - hi).half().float(), hi
    return hi, ops.e4m3_roundtrip(x - hi, ops.ACT_SL8), ops.e4m3_roundtrip(x, ops.ACT_S8)


def _expected(x, wp, conv, P):
    """plain PyTorch fp32 convolution(s) of the SAME rounded operands the kernel multiplies."""
    xm, xl, xa = _operand_terms(x, P)
    wm, wl_for_lo, wlo = wp.effective()
    y = conv(xm, wm)
    if P != 1:
        y = y + conv(xl, wl_for_lo) + conv(xa, wlo)
    return y


def _unpack(m, Cin, Cout, mode, k):
    """packed (rows_total, K) -> the reference's weight layout"""
    if mode == 2:
        kidx = {0: (1, 3), 1: (0, 2)}
        wt = torch.zeros(Cin, Cout, 4, 4)
        for py in range(2):
            for px in range(2):
                blk = m[(py * 2 + px) * Cout:(py * 2 + px + 1) * Cout]
                for ta in range(2):
                    for tb in range(2):
                        wt[:, :, kidx[py][ta], kidx[px][tb]] = blk[:, (ta * 2 + tb) * Cin:(ta * 2 + tb + 1) * Cin].t()
        return wt
    return m.reshape(Cout, k, k, Cin).permute(0, 3, 1, 2).contiguous()


def _planes_problem(N, H, W, Cin, Cout, mode, k, P):
    """seeded operands of a CASES row and the fp32 reference of the rounded operands: (x, w, bias, exp, atol, rtol)"""
    from ipercore_b200 import ops
    x = _rand((N, Cin, H, W), 1)
    wshape = (Cin, Cout, 4, 4) if mode == 2 else (Cout, Cin, k, k)
    fan = Cin * (4 if mode == 2 else k * k)
    w = _rand(wshape, 2, scale=(3.0 / fan) ** 0.5)
    bias = _rand((Cout,), 3, 0.1)
    wp = (ops.pack_convT_weight if mode == 2 else ops.pack_conv_weight)(w, P)

    class _W:
        def effective(self_inner):
            return tuple(None if t is None else _unpack(t, Cin, Cout, mode, k) for t in wp.effective())
    exp = F.relu(_expected(x, _W(), lambda xx, ww: _ref_conv(xx, ww, mode, k), P) + bias.view(1, -1, 1, 1))
    # remaining differences: fp32 accumulation order over K (<= 3456 terms), the dropped lo*lo term (P=2), and the
    # precision of the OUTPUT planes themselves (P=1: 11 bits; P=3: ~15 bits; P=2: ~22 bits)
    atol, rtol = {2: (1e-4, 0), 3: (1.5e-4, 1e-4), 1: (5e-4, 1.1e-3)}[P]
    return x, w, bias, exp, atol, rtol


@pytest.mark.parametrize("P", [2, 1, 3])
@pytest.mark.parametrize("N,H,W,Cin,Cout,mode,k", CASES)
def test_conv_gemm_planes(N, H, W, Cin, Cout, mode, k, P):
    from ipercore_b200 import ops
    from ipercore_b200.ops import Planes
    x, w, bias, exp, atol, rtol = _planes_problem(N, H, W, Cin, Cout, mode, k, P)
    a = Planes.from_nchw(x.to(DEV), P)
    wp = (ops.pack_convT_weight if mode == 2 else ops.pack_conv_weight)(w, P).to(DEV)
    oH, oW = (H // 2, W // 2) if mode == 1 else ((2 * H, 2 * W) if mode == 2 else (H, W))
    out = Planes.empty(P, N, oH, oW, Cout, DEV)
    rows = Cout
    ops.conv_gemm(a, wp, mode, k, rows, 256 if rows >= 256 else rows, ops.IPER_EPI_PLANES, bias=bias.to(DEV), relu=True,
                  out=out)
    torch.cuda.synchronize()
    unpack = lambda m: _unpack(m, Cin, Cout, mode, k)
    got = _planes_value(out)
    np.testing.assert_allclose(got.numpy(), exp.numpy(), atol=atol, rtol=rtol)
    if P != 3:      # both CTA shapes: one or two 128-pixel M tiles per weight tile (K stages of 64 / 32 channels)
        for tm in (1, 2):
            alt = Planes.empty(P, N, oH, oW, Cout, DEV)
            ops.conv_gemm(a, wp, mode, k, rows, 256 if rows >= 256 else rows, ops.IPER_EPI_PLANES, bias=bias.to(DEV),
                          relu=True, out=alt, tiles_m=tm)
            np.testing.assert_allclose(_planes_value(alt).numpy(), exp.numpy(), atol=atol, rtol=rtol)
        if rows >= 128:     # CTA pairs (cta_group::2): the weight tile is split across two SMs
            alt = Planes.empty(P, N, oH, oW, Cout, DEV)
            ops.conv_gemm(a, wp, mode, k, rows, 256 if rows >= 256 else rows, ops.IPER_EPI_PLANES, bias=bias.to(DEV),
                          relu=True, out=alt, cta_pair=1)
            torch.cuda.synchronize()
            np.testing.assert_allclose(_planes_value(alt).numpy(), exp.numpy(), atol=atol, rtol=rtol)
    if _halo_ok(mode, k, 256 if rows >= 256 else rows, H, W):     # vertical taps share one TMA box; fused convT phases
        alt = Planes.empty(P, N, oH, oW, Cout, DEV)
        alt.data.fill_(7.0)
        ops.conv_gemm(a, wp, mode, k, rows, 256 if rows >= 256 else rows, ops.IPER_EPI_PLANES, bias=bias.to(DEV),
                      relu=True, out=alt, cta_pair=2)
        torch.cuda.synchronize()
        np.testing.assert_allclose(_planes_value(alt).numpy(), exp.numpy(), atol=atol, rtol=rtol)
    # on-device cross-check (CUDA-core direct convolution of the stored activation values with the fp16-rounded weights)
    chk = Planes.empty(P, N, oH, oW, Cout, DEV)
    wm, _, wlo = wp.effective()
    w_total = wm if wlo is None else wm + wlo            # the weight value the MMA groups add up to
    ops.conv_direct(a, unpack(w_total).to(DEV), mode, k, Cout, ops.IPER_EPI_PLANES, bias=bias.to(DEV), relu=True, out=chk)
    np.testing.assert_allclose(got.numpy(), _planes_value(chk).numpy(), atol={2: 2e-4, 3: 4e-4, 1: 5e-4}[P],
                               rtol={2: 0, 3: 1e-4, 1: 1.1e-3}[P])


def test_conv_gemm_fp32_out_residual_and_windows():
    """EPI_F32 (q / kv projections), residual add, channel windows of wider buffers (decoder concatenations)."""
    from ipercore_b200 import ops
    from ipercore_b200.ops import Planes
    P, N, H, W = 2, 2, 16, 16
    x = _rand((N, 128, H, W), 11)
    w = _rand((256, 128, 1, 1), 12, 0.1); b = _rand((256,), 13, 0.1)
    buf = Planes.empty(P, N, H, W, 320, DEV); buf.data.zero_()
    a = Planes.from_nchw(x.to(DEV), P, out=buf.window(64, 128))
    xq = _planes_value(a)
    out = torch.empty((N, H, W, 256), dtype=torch.float32, device=DEV)
    ops.conv_gemm(a, ops.pack_conv_weight(w, P).to(DEV), 0, 1, 256, 256, ops.IPER_EPI_F32, bias=b.to(DEV), out=out)
    exp = F.conv2d(xq, ops.split_planes(w, P).float().sum(0)) + b.view(1, -1, 1, 1)
    np.testing.assert_allclose(out.permute(0, 3, 1, 2).cpu().numpy(), exp.numpy(), atol=2e-5, rtol=0)
    # residual: y = x + conv3x3(x) written into a window
    w3 = _rand((128, 128, 3, 3), 14, 0.03)
    dst = Planes.empty(P, N, H, W, 384, DEV); dst.data.zero_()
    ops.conv_gemm(a, ops.pack_conv_weight(w3, P).to(DEV), 0, 3, 128, 128, ops.IPER_EPI_PLANES, bias=None, relu=False,
                  out=dst.window(128, 128), x=a)
    exp = xq + F.conv2d(xq, ops.split_planes(w3, P).float().sum(0), padding=1)
    np.testing.assert_allclose(_planes_value(dst.window(128, 128)).numpy(), exp.numpy(), atol=3e-5, rtol=0)
    assert float(dst.window(0, 128).to_nchw().abs().max()) == 0.0 and float(dst.window(256, 128).to_nchw().abs().max()) == 0.0


@pytest.mark.parametrize("C,P", [(64, 2), (128, 2), (256, 2), (256, 1), (128, 3), (256, 3)])
def test_conv_gemm_spade_epilogue(C, P):
    """mlp_gamma|mlp_beta GEMM fused with IN(x)*(1+gamma)+beta (attlwb_spade_resunet.py:80-93)."""
    from ipercore_b200 import ops
    from ipercore_b200.ops import Planes
    N, H, W = 2, 16, 16
    actv = F.relu(_rand((N, 128, H, W), 21)); x = F.relu(_rand((N, C, H, W), 22) + 0.3)
    wg = _rand((C, 128, 3, 3), 23, 0.02); wb = _rand((C, 128, 3, 3), 24, 0.02); bg = _rand((C,), 25, 0.1); bb = _rand((C,), 26, 0.1)
    a = Planes.from_nchw(actv.to(DEV), P); xp = Planes.from_nchw(x.to(DEV), P)
    aq, xq = _planes_value(a), _planes_value(xp)
    stats = ops.instnorm_stats(xp)
    bn = 256 if 2 * C >= 256 else 2 * C
    wpk, bpk = ops.pack_spade_weight(wg, bg, wb, bb, P, bn)
    out = Planes.empty(P, N, H, W, C, DEV)
    ops.conv_gemm(a, wpk.to(DEV), 0, 3, 2 * C, bn, ops.IPER_EPI_SPADE, bias=bpk.to(DEV), out=out, x=xp, mean_rstd=stats,
                  spade_C=C)
    q = lambda t: ops.split_planes(t, P).float().sum(0)        # fp16-rounded weights (hi+lo for P=2)
    gamma = F.conv2d(aq, q(wg), bg, padding=1); beta = F.conv2d(aq, q(wb), bb, padding=1)
    exp = F.instance_norm(xq, eps=1e-5) * (1 + gamma) + beta
    mean = xq.mean((2, 3)); var = xq.var((2, 3), unbiased=False)
    np.testing.assert_allclose(stats[..., 0].cpu().numpy(), mean.numpy(), atol=1e-6, rtol=0)
    np.testing.assert_allclose(stats[..., 1].cpu().numpy(), (1 / torch.sqrt(var + 1e-5)).numpy(), rtol=2e-6, atol=0)
    np.testing.assert_allclose(_planes_value(out).numpy(), exp.numpy(), atol={2: 1e-4, 3: 1.5e-3, 1: 3e-3}[P], rtol=0)
    for mode_pair in ((1, 2) if bn >= 128 else (2,)) if P != 3 else (2,):      # CTA pair, CTA pair + halo
        alt = Planes.empty(P, N, H, W, C, DEV)
        ops.conv_gemm(a, wpk.to(DEV), 0, 3, 2 * C, bn, ops.IPER_EPI_SPADE, bias=bpk.to(DEV), out=alt, x=xp,
                      mean_rstd=stats, spade_C=C, cta_pair=mode_pair)
        np.testing.assert_allclose(_planes_value(alt).numpy(), exp.numpy(), atol={2: 1e-4, 3: 1.5e-3, 1: 3e-3}[P], rtol=0)
    chk = Planes.empty(P, N, H, W, C, DEV)
    ops.conv_direct(a, torch.cat([q(wg), q(wb)], 0).to(DEV), 0, 3, 2 * C, ops.IPER_EPI_SPADE, bias=torch.cat([bg, bb]).to(DEV),
                    out=chk, x=xp, mean_rstd=stats, spade_C=C)
    np.testing.assert_allclose(_planes_value(chk).numpy(), exp.numpy(), atol={2: 1e-4, 3: 1.5e-3, 1: 3e-3}[P], rtol=0)


def _heads_problem(S, P):
    """seeded heads operands and the fp32 reference: (x, wi, wm, bgimg, ei, em, tol)"""
    from ipercore_b200 import ops
    from ipercore_b200.ops import Planes
    N = 2
    x = F.relu(_rand((N, 64, S, S), 31)); wi = _rand((3, 64, 5, 5), 32, 0.03); wm = _rand((1, 64, 5, 5), 33, 0.03)
    bgimg = _rand((1, 3, S, S), 34)
    xq = _planes_value(Planes.from_nchw(x.to(DEV), P))
    q = lambda t: ops.split_planes(t, P).float().sum(0)
    ei = torch.tanh(F.conv2d(xq, q(wi), padding=2)); em = torch.sigmoid(F.conv2d(xq, q(wm), padding=2))
    return x, wi, wm, bgimg, ei, em, {2: 3e-5, 3: 3e-4, 1: 2e-3}[P]


def _check_heads(img, mask, pred, ei, em, bgimg, tol, label):
    for name, got, exp, t in (("img", img, ei, tol), ("mask", mask, em, tol), ("pred", pred, em * bgimg + (1 - em) * ei, 1.5 * tol)):
        got = torch.as_tensor(got).cpu()
        print("%s %s: max |err| %.2e" % (label, name, float((got - exp).abs().max())))
        np.testing.assert_allclose(got.numpy(), exp.numpy(), atol=t, rtol=0)


@pytest.mark.parametrize("S,P", [(32, 2), (300, 2), (300, 3), (64, 1)])
def test_conv_gemm_heads_epilogue(S, P):
    """5x5 heads (64->3 tanh, 64->1 sigmoid) + composite (imitator.py:393)."""
    from ipercore_b200 import ops
    from ipercore_b200.ops import Planes
    N = 2
    x, wi, wm, bgimg, ei, em, tol = _heads_problem(S, P)
    a = Planes.from_nchw(x.to(DEV), P)
    wp = ops.pack_heads_weight(wi, wm, P).to(DEV)
    img = torch.empty((N, 3, S, S), device=DEV); mask = torch.empty((N, 1, S, S), device=DEV); pred = torch.empty((N, 3, S, S), device=DEV)
    ops.conv_gemm(a, wp, ops.IPER_CONV_ROW5, 5, 32, 32, ops.IPER_EPI_HEADS, heads=dict(img=img, mask=mask, pred=pred, bg=bgimg.to(DEV)))
    _check_heads(img, mask, pred, ei, em, bgimg, tol, "heads S=%d P=%d" % (S, P))
    # halo kernel: 32x4 tiles, the five vertical taps are views of one 32x8 box (with P=2: the N-concatenated
    # [w_hi ; w_lo] form, 2 MMAs per K step; the 3-MMA form runs in test_heads_three_mma_form)
    img2 = torch.full_like(img, 9.0); mask2 = torch.full_like(mask, 9.0); pred2 = torch.full_like(pred, 9.0)
    ops.conv_gemm(a, wp, ops.IPER_CONV_ROW5, 5, 32, 32, ops.IPER_EPI_HEADS,
                  heads=dict(img=img2, mask=mask2, pred=pred2, bg=bgimg.to(DEV)), cta_pair=2)
    _check_heads(img2, mask2, pred2, ei, em, bgimg, tol, "heads halo S=%d P=%d" % (S, P))


# ----------------------------------------------------------------------------------------------------------------------
# IPER_HEADS_CAT=0 / IPER_CONVT_FUSE_N=0: read once per process by the library, so they run in one child process
# ----------------------------------------------------------------------------------------------------------------------
HEADS_3MMA = [(32, 2), (300, 2)]
# the mode-2 rows of CASES the halo (cta_pair = 2) kernel takes: the only kernel with fused transposed-conv phases
CONVT_UNFUSED = [(c, P) for c in CASES if c[5] == 2 and _halo_ok(2, 4, 256 if c[4] >= 256 else c[4], c[1], c[2]) for P in (1, 2)]
VARIANT_ENV = {"IPER_HEADS_CAT": "0", "IPER_CONVT_FUSE_N": "0"}


def child_heads_convt(inputs):
    """the halo kernel on the HEADS_3MMA and CONVT_UNFUSED problems (this process's switches)"""
    from ipercore_b200 import ops
    from ipercore_b200.ops import Planes
    t = lambda k: torch.from_numpy(inputs[k])
    out = {}
    for S, P in HEADS_3MMA:
        a = Planes.from_nchw(t("h%d_%d_x" % (S, P)).to(DEV), P)
        wp = ops.pack_heads_weight(t("h%d_%d_wi" % (S, P)), t("h%d_%d_wm" % (S, P)), P).to(DEV)
        hd = {k: torch.full((2, c, S, S), 9.0, device=DEV) for k, c in (("img", 3), ("mask", 1), ("pred", 3))}
        ops.conv_gemm(a, wp, ops.IPER_CONV_ROW5, 5, 32, 32, ops.IPER_EPI_HEADS,
                      heads=dict(hd, bg=t("h%d_%d_bg" % (S, P)).to(DEV)), cta_pair=2)
        out.update({"h%d_%d_%s" % (S, P, k): v.cpu().numpy() for k, v in hd.items()})
    for i, ((N, H, W, Cin, Cout, mode, k), P) in enumerate(CONVT_UNFUSED):
        a = Planes.from_nchw(t("c%d_x" % i).to(DEV), P)
        wp = ops.pack_convT_weight(t("c%d_w" % i), P).to(DEV)
        o = Planes.empty(P, N, 2 * H, 2 * W, Cout, DEV)
        o.data.fill_(7.0)
        ops.conv_gemm(a, wp, mode, k, Cout, Cout, ops.IPER_EPI_PLANES, bias=t("c%d_b" % i).to(DEV), relu=True, out=o,
                      cta_pair=2)
        out["c%d_out" % i] = o.to_nchw().cpu().numpy()
    torch.cuda.synchronize()
    return out


@pytest.fixture(scope="module")
def variant_outputs(tmp_path_factory):
    from test_attention_gpu import run_variant
    inputs = {}
    for S, P in HEADS_3MMA:
        x, wi, wm, bgimg = _heads_problem(S, P)[:4]
        inputs.update({"h%d_%d_x" % (S, P): x.numpy(), "h%d_%d_wi" % (S, P): wi.numpy(), "h%d_%d_wm" % (S, P): wm.numpy(),
                       "h%d_%d_bg" % (S, P): bgimg.numpy()})
    for i, (case, P) in enumerate(CONVT_UNFUSED):
        x, w, bias = _planes_problem(*case, P)[:3]
        inputs.update({"c%d_x" % i: x.numpy(), "c%d_w" % i: w.numpy(), "c%d_b" % i: bias.numpy()})
    out, kernels = run_variant(tmp_path_factory.mktemp("variants"), VARIANT_ENV, "test_conv_gpu", "child_heads_convt", inputs)
    print("child with %s ran: %s" % (VARIANT_ENV, ", ".join(sorted({n.split("(")[0] for n in kernels}))))
    return out


@pytest.mark.parametrize("S,P", HEADS_3MMA)
def test_heads_three_mma_form(S, P, variant_outputs):
    """IPER_HEADS_CAT=0: the halo heads kernel with three MMAs per K step (hi*w_hi, hi*w_lo, lo*w_hi) instead of the
    N-concatenated weights, against the same reference and tolerance as the default form"""
    x, wi, wm, bgimg, ei, em, tol = _heads_problem(S, P)
    g = lambda k: torch.from_numpy(variant_outputs["h%d_%d_%s" % (S, P, k)])
    _check_heads(g("img"), g("mask"), g("pred"), ei, em, bgimg, tol, "heads 3-MMA (IPER_HEADS_CAT=0) S=%d P=%d" % (S, P))


@pytest.mark.parametrize("case,P", CONVT_UNFUSED, ids=lambda v: str(v))
def test_convT_unfused_phases(case, P, variant_outputs):
    """IPER_CONVT_FUSE_N=0: the halo kernel's transposed convolution with one MMA group per phase, against the
    reference test_conv_gemm_planes uses"""
    i = CONVT_UNFUSED.index((case, P))
    exp, atol, rtol = _planes_problem(*case, P)[3:]
    got = variant_outputs["c%d_out" % i]
    print("convT unfused %s P=%d: max |err| %.2e" % (case, P, float(np.abs(got - exp.numpy()).max())))
    np.testing.assert_allclose(got, exp.numpy(), atol=atol, rtol=rtol)


def test_stem_direct_kernel():
    """the CUDA-core stem (IPER_STEM=direct); iper_warp_attention is tested in test_attention_gpu.py"""
    from ipercore_b200 import ops
    from ipercore_b200.ops import Planes
    P, N, S = 2, 2, 64
    x = _rand((N, 6, S, S), 41); w = _rand((64, 6, 3, 3), 42, 0.2); b = _rand((64,), 43, 0.1)
    out = Planes.empty(P, N, S // 2, S // 2, 64, DEV)
    ops.conv_stem(x.to(DEV), w.to(DEV), b.to(DEV), out)
    exp = F.relu(F.conv2d(x, w, b, stride=2, padding=1))
    np.testing.assert_allclose(_planes_value(out).numpy(), exp.numpy(), atol=1e-5, rtol=0)


@pytest.mark.parametrize("N,H,W,Cin,Cout,mode", [(3, 16, 16, 64, 128, 0), (2, 32, 32, 64, 128, 1), (5, 4, 4, 128, 256, 0)])
def test_fused_instnorm_statistics(N, H, W, Cin, Cout, mode):
    """statistics fused into the producing conv (+residual/ReLU) == statistics of the stored tensor (stand-alone kernel)."""
    from ipercore_b200 import ops
    from ipercore_b200.ops import Planes
    P = 2
    x = _rand((N, Cin, H, W), 61); w = _rand((Cout, Cin, 3, 3), 62, 0.05); b = _rand((Cout,), 63, 0.2)
    a = Planes.from_nchw(x.to(DEV), P)
    oH, oW = (H // 2, W // 2) if mode == 1 else (H, W)
    out = Planes.empty(P, N, oH, oW, Cout, DEV)
    ws = ops.stats_workspace(N, Cout, DEV)
    ops.conv_gemm(a, ops.pack_conv_weight(w, P).to(DEV), mode, 3, Cout, 256 if Cout >= 256 else Cout, ops.IPER_EPI_PLANES,
                  bias=b.to(DEV), relu=True, out=out, stats_ws=ws)
    fused = ops.instnorm_finalize(ws, oH * oW)
    alone = ops.instnorm_stats(out)
    torch.testing.assert_close(fused[..., 0], alone[..., 0], atol=2e-6, rtol=0)
    torch.testing.assert_close(fused[..., 1], alone[..., 1], atol=0, rtol=2e-5)
    if mode == 0 and H >= 8 and W >= 16:       # the halo kernel shares the epilogue
        ws3 = ops.stats_workspace(N, Cout, DEV)
        ops.conv_gemm(a, ops.pack_conv_weight(w, P).to(DEV), mode, 3, Cout, 256 if Cout >= 256 else Cout, ops.IPER_EPI_PLANES,
                      bias=b.to(DEV), relu=True, out=out, stats_ws=ws3, cta_pair=2)
        f3 = ops.instnorm_finalize(ws3, oH * oW)
        torch.testing.assert_close(f3[..., 0], alone[..., 0], atol=2e-6, rtol=0)
        torch.testing.assert_close(f3[..., 1], alone[..., 1], atol=0, rtol=2e-5)
    # stem
    xi = _rand((N, 6, 2 * H, 2 * W), 64); ws2 = ops.stats_workspace(N, 64, DEV)
    so = Planes.empty(P, N, H, W, 64, DEV)
    ops.conv_stem(xi.to(DEV), _rand((64, 6, 3, 3), 65, 0.2).to(DEV), None, so, stats_ws=ws2)
    f2 = ops.instnorm_finalize(ws2, H * W); a2 = ops.instnorm_stats(so)
    torch.testing.assert_close(f2[..., 0], a2[..., 0], atol=2e-6, rtol=0)
    torch.testing.assert_close(f2[..., 1], a2[..., 1], atol=0, rtol=2e-5)


def test_split_fp16_range_and_small_values():
    """VERDICT r01 weak point 9: the hi/lo planes have fp16 RANGE.  Documented behaviour, probed with adversarial scales:
    values up to 6e4 survive the planes round trip and a convolution at ~22 bits; tiny values are kept to an ABSOLUTE error of
    one fp16 subnormal step (3e-8) — the lo plane underflows, the hi plane does not; beyond 65504 the planes go non-finite
    (the kernels do not clamp: an instance-normalised network never gets there, and a silent clamp would hide a real bug)."""
    from ipercore_b200 import ops
    from ipercore_b200.ops import Planes
    g = torch.Generator().manual_seed(3)
    mag = 10.0 ** (torch.rand((1, 64, 16, 16), generator=g) * 11.5 - 7.0)          # 1e-7 .. 3e4
    x = (mag * torch.sign(torch.rand(mag.shape, generator=g) - 0.5)).clamp(-6.0e4, 6.0e4)
    back = Planes.from_nchw(x.to(DEV), 2).to_nchw().cpu()
    err = (back - x).abs()
    assert torch.isfinite(back).all()
    assert (err <= torch.maximum(x.abs() * 2.0 ** -21, torch.tensor(6.0e-8))).all(), float((err / x.abs()).max())
    # a 3x3 convolution over large-magnitude activations and small weights: fp32 reference of the same math
    xa = (_rand((1, 64, 16, 16), 5) * 3.0e4)
    w = _rand((64, 64, 3, 3), 6, 1e-3)
    wp = ops.pack_conv_weight(w, 2)
    wp.w = wp.w.to(DEV)
    out = Planes.empty(2, 1, 16, 16, 64, DEV)
    ops.conv_gemm(Planes.from_nchw(xa.to(DEV), 2), wp, ops.IPER_CONV_S1, 3, 64, 64, ops.IPER_EPI_PLANES, out=out, cta_pair=0)
    ref = F.conv2d(xa.double(), w.double(), padding=1).float()
    rel = float((out.to_nchw().cpu() - ref).abs().max() / ref.abs().max())
    print("conv over |x| ~ 3e4: relative error %.2e" % rel)
    assert rel <= 4e-6          # 2.4e-5 without the power-of-two weight pre-scale (the lo plane of 1e-3 weights is subnormal)
    over = Planes.from_nchw(torch.full((1, 8, 8, 8), 7.0e4, device=DEV), 2).to_nchw()
    assert not torch.isfinite(over).any()                # loud, not silent: hi = inf, lo = x - inf -> the value reads back non-finite


@pytest.mark.parametrize("N,H,W,P", [(2, 64, 64, 2), (3, 40, 72, 2), (1, 16, 32, 1), (5, 512, 512, 2)])
def test_stem_tensor_core_forms(N, H, W, P):
    """First encoder layer (Conv2d(6, 64, 3, s2, p1) + bias + ReLU, attlwb_spade_resunet.py:268-271) in its three forms:
    iper_conv_stem_tc (A operand built in shared memory by builder warps — the default), im2col + 1x1 GEMM, and the CUDA-core
    kernel, against torch fp32; partial tiles (20x36 output), a 256^2 output with several images per CTA range, single plane;
    the fused instance-norm sums against a separate statistics pass."""
    from ipercore_b200 import ops
    from ipercore_b200.ops import Planes
    x = _rand((N, 6, H, W), 71); w = _rand((64, 6, 3, 3), 72, 0.2); b = _rand((64,), 73, 0.1)
    exp = F.relu(F.conv2d(x, w, b, stride=2, padding=1))
    tol = 1e-5 if P == 2 else 5e-3
    wp = ops.pack_stem_weight(w.to(DEV), P)
    out = Planes.empty(P, N, H // 2, W // 2, 64, DEV)
    ws = ops.stats_workspace(N, 64, DEV)
    ops.conv_stem_tc(x.to(DEV), wp, b.to(DEV), out, stats_ws=ws)
    got = _planes_value(out)
    print("stem tc %s P=%d: max err %.2e" % ((N, H, W), P, float((got - exp).abs().max())))
    np.testing.assert_allclose(got.numpy(), exp.numpy(), atol=tol, rtol=0)
    # fused sums are taken from the fp32 values before the planes store; a single fp16 plane (P = 1) then differs by its rounding
    sa, sr = (2e-6, 2e-5) if P == 2 else (1e-4, 1e-3)
    f, a = ops.instnorm_finalize(ws, (H // 2) * (W // 2)), ops.instnorm_stats(out)
    torch.testing.assert_close(f[..., 0], a[..., 0], atol=sa, rtol=0)
    torch.testing.assert_close(f[..., 1], a[..., 1], atol=0, rtol=sr)
    if H <= 128:
        col = Planes.empty(P, N, H // 2, W // 2, 64, DEV)
        ops.stem_im2col(x.to(DEV), col)
        out2 = Planes.empty(P, N, H // 2, W // 2, 64, DEV)
        ws2 = ops.stats_workspace(N, 64, DEV)
        ops.conv_gemm(col, wp, ops.IPER_CONV_S1, 1, 64, 64, ops.IPER_EPI_PLANES, bias=b.to(DEV), relu=True, out=out2, stats_ws=ws2)
        np.testing.assert_allclose(_planes_value(out2).numpy(), exp.numpy(), atol=tol, rtol=0)
        f2 = ops.instnorm_finalize(ws2, (H // 2) * (W // 2))     # per-warp running sums of conv_gemm_kernel
        torch.testing.assert_close(f2[..., 0], a[..., 0], atol=sa, rtol=0)
        torch.testing.assert_close(f2[..., 1], a[..., 1], atol=0, rtol=sr)
        out3 = Planes.empty(P, N, H // 2, W // 2, 64, DEV)
        ops.conv_stem(x.to(DEV), w.to(DEV), b.to(DEV), out3)
        np.testing.assert_allclose(_planes_value(out3).numpy(), exp.numpy(), atol=tol, rtol=0)
