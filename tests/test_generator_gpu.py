"""GPU parity of the generator path (seam B3) against the golden fixtures produced by the REFERENCE's own
AttentionLWBGenerator on CPU in fp32 (tests/golden/make_golden.py).  Tolerance: BASELINE.json north_star —
1e-3 max-abs for the fp32-parity mode ("fp16x2")."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

CFG = dict(name="AttLWB-SPADE", BGNet=dict(cond_nc=4, n_res_block=6, num_filters=[64, 128, 128, 256]),
           SIDNet=dict(cond_nc=6, n_res_block=6, num_filters=[64, 128, 256]),
           TSFNet=dict(cond_nc=6, n_res_block=6, num_filters=[64, 128, 256]))


def _gen(precision):
    from ipercore_b200.generator import AttentionLWBGenerator
    from oracle.weights import synth_state_dict
    g = AttentionLWBGenerator(CFG, precision=precision)
    g.load_state_dict(synth_state_dict(0), strict=True)
    return g.to("cuda:0").eval()


@pytest.mark.parametrize("S,precision,tol", [(256, "fp16x2", 1e-3), (64, "fp16x2", 1e-3), (256, "fp16f8", 1e-3),
                                             (64, "fp16f8", 1e-3), (256, "fp16", 1e-2),
                                             # single-plane SPADE convolutions: 6.6e-4 .. 1.8e-3 in the CPU emulation
                                             # (tools/precision_plan.py); not a 1e-3 mode
                                             (256, "mixed", 3e-3)])
def test_forward_src_tsf_matches_reference(S, precision, tol, golden_dir):
    import make_golden
    g = np.load(os.path.join(golden_dir, "gen_S%d.npz" % S))
    inp = {k: torch.from_numpy(v).to("cuda:0") for k, v in make_golden.gen_inputs(S).items()}
    net = _gen(precision)
    enc, res = net.forward_src(inp["src_inputs"], only_enc=True)
    img, mask = net.forward_tsf(inp["tsf_inputs"], enc, res, inp["Tst"])
    torch.cuda.synchronize()
    e_enc = np.abs(enc[2].cpu().numpy() - g["src_enc2"]).max()
    e_res = np.abs(res[5].cpu().numpy() - g["src_res5"]).max()
    e_img = np.abs(img.cpu().numpy() - g["tsf_img"]).max()
    e_mask = np.abs(mask.cpu().numpy() - g["tsf_mask"]).max()
    print("S=%d %s: max-abs err src_enc2 %.2e src_res5 %.2e tsf_img %.2e tsf_mask %.2e" % (S, precision, e_enc, e_res, e_img, e_mask))
    assert e_img <= tol and e_mask <= tol, (e_img, e_mask)
    assert e_enc <= tol and e_res <= tol, (e_enc, e_res)      # measured 2e-5 / 7e-5 in fp16x2


def test_batched_frames_equal_single_frames(golden_dir):
    """Frames are independent: a batch of B frames equals B single-frame calls."""
    import make_golden
    S = 128
    inp = {k: torch.from_numpy(v).to("cuda:0") for k, v in make_golden.gen_inputs(S).items()}
    net = _gen("fp16x2")
    enc, res = net.forward_src(inp["src_inputs"], only_enc=True)
    tsf = torch.cat([inp["tsf_inputs"], inp["tsf_inputs"].flip(-1), inp["tsf_inputs"] * 0.5], 0)
    Tst = torch.cat([inp["Tst"], inp["Tst"].flip(2), inp["Tst"]], 0).contiguous()
    bg = torch.rand(1, 3, S, S, device="cuda:0") * 2 - 1
    img, mask, pred = net.forward_tsf(tsf, enc, res, Tst, bg_img=bg, return_pred=True)
    for i in range(3):
        im1, m1 = net.forward_tsf(tsf[i:i + 1].contiguous(), enc, res, Tst[i:i + 1].contiguous())
        # instance-norm sums are fp64 atomics (order-dependent in the last fp64 bits); everything else is deterministic
        d = max(float((im1[0] - img[i]).abs().max()), float((m1[0] - mask[i]).abs().max()))
        print("batched vs single frame %d: max diff %.3e" % (i, d))
        assert d <= 1e-5
    torch.testing.assert_close(pred, mask * bg + (1 - mask) * img, atol=1e-6, rtol=0)


def test_forward_bg_matches_reference(golden_dir):
    """BGNet (bg_inpaintor.py:24-60), one-time per source: conv7x7 / IN / ReLU / s2 convs / res blocks / convT / tanh."""
    import make_golden
    S = 64
    g = np.load(os.path.join(golden_dir, "gen_S%d.npz" % S))
    inp = make_golden.gen_inputs(S)
    net = _gen("fp16x2")
    bg = net.forward_bg(torch.from_numpy(inp["bg_inputs"]).to("cuda:0"))
    torch.cuda.synchronize()
    err = np.abs(bg.cpu().numpy() - g["bg_img"]).max()
    print("forward_bg max-abs err %.2e" % err)
    assert bg.shape == (1, 1, 3, S, S) and err <= 1e-3


@pytest.mark.parametrize("S,ns,B", [(192, 3, 2), (320, 1, 1)])
def test_generic_sizes_and_source_counts(S, ns, B, template):
    """Sizes that are not powers of two (partial tiles at every level) and ns != 2, whole path vs the CPU oracle."""
    from ipercore_b200.renders import SMPLRenderer
    from oracle import flow_ref, generator_ref, synth, weights
    dev = "cuda:0"
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    sd = weights.synth_state_dict(0)
    net = _gen("fp16x2")
    r = SMPLRenderer(image_size=S, tables=template).to(dev)
    cams, verts = synth.pose_sweep(template, B, total=9, start=1)
    scams, sverts = synth.source_views(template, ns)
    uv_img = synth.smooth_image((1, 3, S, S), seed=21); src_img = synth.smooth_image((ns, 3, S, S), seed=22)
    src_f2pts, sfim, _ = flow_ref.render_fim_wim(scams, sverts, template["faces"], S)
    src_inputs = np.concatenate([src_img, flow_ref.encode_fim(sfim, template["map_fn"])], 1)[None]
    want = flow_ref.frame_inputs(cams, verts, template["faces"], template["map_fn"], template["f_uvs2img"], uv_img,
                                 src_f2pts, S)
    got = r.frame_inputs(t(cams), t(verts), t(uv_img), t(src_f2pts), want_fim=True)
    np.testing.assert_array_equal(got["fim"].cpu().numpy(), want["fim"])
    np.testing.assert_allclose(got["Tst"].cpu().numpy(), want["Tst"], atol=1e-6, rtol=0)
    enc, res = net.forward_src(t(src_inputs))
    img, mask = net.forward_tsf(got["tsf_inputs"], enc, res, got["Tst"])
    err = 0.0
    with torch.no_grad():
        se, sr = generator_ref.forward_src(sd, torch.from_numpy(src_inputs))
        for i in range(B):
            ei, em = generator_ref.forward_tsf(sd, torch.from_numpy(want["tsf_inputs"][i:i + 1]), se, sr,
                                               torch.from_numpy(want["Tst"][i:i + 1]))
            err = max(err, float((img[i:i + 1].cpu() - ei).abs().max()), float((mask[i:i + 1].cpu() - em).abs().max()))
    print("S=%d ns=%d: max-abs err %.2e" % (S, ns, err))
    assert err <= 1e-3


def test_temporal_attention_matches_reference_golden(golden_dir):
    """temporal=True (attlwb_spade_resunet.py:208-252, 480-535): the previous frame's features are extra attention sources with
    their own flow Ttt — vs the reference generator built with temporal=True (tests/golden/gen_S64_temporal.npz)."""
    import make_golden
    from ipercore_b200.generator import AttentionLWBGenerator
    from oracle.weights import synth_state_dict
    S = 64
    g = np.load(os.path.join(golden_dir, "gen_S%d_temporal.npz" % S))
    inp = {k: torch.from_numpy(v).to("cuda:0") for k, v in make_golden.gen_inputs(S).items()}
    prev, Ttt = (torch.from_numpy(a).to("cuda:0") for a in make_golden.temporal_inputs(S))
    net = AttentionLWBGenerator(CFG, temporal=True); net.load_state_dict(synth_state_dict(0), strict=True); net = net.to("cuda:0").eval()
    enc, res = net.forward_src(inp["src_inputs"], only_enc=True)
    tenc, tres = net.forward_src(prev, only_enc=True)
    img, mask = net.forward_tsf(inp["tsf_inputs"], enc, res, inp["Tst"], tenc, tres, Ttt)
    e = max(np.abs(img.cpu().numpy() - g["tsf_img"]).max(), np.abs(mask.cpu().numpy() - g["tsf_mask"]).max())
    img0, _ = net.forward_tsf(inp["tsf_inputs"], enc, res, inp["Tst"])
    print("temporal forward_tsf vs reference: %.2e (the temporal source moves the output by %.2f)" % (e, float((img - img0).abs().max())))
    assert e <= 1e-3 and float((img - img0).abs().max()) > 0.05
    with pytest.raises(NotImplementedError, match="bs = 1"):
        net.forward_tsf(inp["tsf_inputs"].repeat(2, 1, 1, 1), enc, res, inp["Tst"].repeat(2, 1, 1, 1, 1), tenc, tres, Ttt.repeat(2, 1, 1, 1, 1))
