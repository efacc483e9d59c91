"""CPU tests of the C-ABI boundary: the library builds/loads, exports every symbol include/iper_b200.h declares,
argument validation reports errors (no compute is launched without a GPU), and the host-side module keeps the
reference's checkpoint layout."""
import ctypes
import os
import re

import pytest
import torch

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))


def _declared_symbols():
    hdr = open(os.path.join(ROOT, "include", "iper_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    return sorted(set(re.findall(r"\b(iper_[a-z0-9_]+)\s*\(", hdr)))


def test_library_exports_every_declared_symbol():
    from ipercore_b200 import _lib
    names = _declared_symbols()
    assert len(names) >= 15
    raw = ctypes.CDLL(_lib.LIB_PATH)
    for n in names:
        assert hasattr(raw, n), "libiper_b200.so does not export %s" % n
    assert set(_lib.SIGNATURES) | set(_lib.OTHER_SIGNATURES) == set(names), "ctypes table and header drifted apart"
    assert _lib.lib.iper_abi_version() == 1


def test_descriptor_struct_matches_header():
    from ipercore_b200._lib import ConvGemmDesc
    assert ctypes.sizeof(ConvGemmDesc) == 288 and ConvGemmDesc.w_scale_inv.offset == 280 and ConvGemmDesc.cta_pair.offset == 272 and ConvGemmDesc.tiles_m.offset == 260 and ConvGemmDesc.stats_ws.offset == 264 and ConvGemmDesc.max_ctas.offset == 232 and ConvGemmDesc.cross_scale.offset == 256


def test_adam_segment_struct_matches_header():
    from ipercore_b200._lib import AdamSeg
    assert ctypes.sizeof(AdamSeg) == 56 and AdamSeg.taps.offset == 24 and AdamSeg.fwd_offset.offset == 40 and AdamSeg.dgrad_offset.offset == 48


def test_argument_validation_reports_errors():
    from ipercore_b200 import _lib
    d = _lib.ConvGemmDesc()
    assert _lib.lib.iper_conv_gemm(ctypes.byref(d), None) != 0
    assert b"null" in _lib.lib.iper_last_error()
    with pytest.raises(RuntimeError, match="iper_b200"):
        _lib.check(_lib.lib.iper_rasterize_faces(None, 1, 1, 8, 0.1, 100.0, None, None, None, 0, None), "rasterize_faces")


def test_training_entry_points_validate_arguments():
    """The training-step entry points reject bad arguments with a status and a message before touching the device."""
    from ipercore_b200 import _lib
    L = _lib.lib
    assert L.iper_conv_bf16(None, 1, 64, 64, 64, None, 64, 3, 1, 1, None, 0, None, None, None) != 0 and b"null" in L.iper_last_error()
    assert L.iper_conv_bf16(16, 1, 64, 64, 64, 16, 64, 9, 1, 1, None, 0, None, 16, None) != 0 and b"kernel 9" in L.iper_last_error()
    assert L.iper_conv_bf16(16, 1, 64, 64, 60, 16, 64, 3, 1, 1, None, 0, None, 16, None) != 0 and b"Cin" in L.iper_last_error()
    assert L.iper_conv_bf16(16, 1, 63, 64, 64, 16, 64, 3, 2, 1, None, 0, None, 16, None) != 0 and b"even" in L.iper_last_error()
    assert L.iper_conv_bf16(16, 1, 4, 64, 64, 16, 64, 3, 1, 1, None, 0, None, 16, None) != 0 and b"too small" in L.iper_last_error()
    assert L.iper_conv_transposed_bf16(16, 1, 16, 16, 64, 16, 64, 5, 1, None, 0, 16, None) != 0 and b"kernel 5" in L.iper_last_error()
    assert L.iper_conv_wgrad_bf16(16, 16, 1, 64, 64, 64, 64, 3, 1, 1, None, 1, 1, 1, 64, 64, None) != 0 and b"null" in L.iper_last_error()
    assert L.iper_conv_wgrad_bf16(16, 16, 1, 64, 64, 64, 64, 3, 1, 1, 16, 1, 1, 1, 65, 64, None) != 0 and b"valid channel" in L.iper_last_error()
    assert L.iper_bias_grad_bf16(16, 10, 70, 64, 16, None) != 0 and b"pitch" in L.iper_last_error()
    assert L.iper_thin_wgrad_bf16(16, 16, 1, 64, 64, 64, 64, 5, 5, 2, 1, 16, 1, 1, 1, None) != 0 and b"Ct" in L.iper_last_error()
    assert L.iper_att_combine_bf16(16, 16, 16, 1, 9, 64, 64, 16, 16, None) != 0 and b"ns" in L.iper_last_error()
    assert L.iper_norm_stats_bf16(16, 1, 64, 72, 16, None) != 0 and b"unsupported C" in L.iper_last_error()
    assert L.iper_pad_nhwc_bf16(16, 0, 1, 6, 8, 8, 384, 64, 8, 1, 60, 16, None) != 0 and b"Cpad" in L.iper_last_error()
    assert L.iper_adam_pack(None, None, None, None, None, None, 0, 0, 1e-4, 0.9, 0.999, 1e-8, 1.0, None, 1, None, None, None) != 0


def test_generator_loads_reference_checkpoint_layout():
    from ipercore_b200.generator import AttentionLWBGenerator
    from oracle.weights import synth_state_dict
    cfg = dict(name="AttLWB-SPADE", BGNet=dict(cond_nc=4, n_res_block=6, num_filters=[64, 128, 128, 256]),
               SIDNet=dict(cond_nc=6, n_res_block=6, num_filters=[64, 128, 256]),
               TSFNet=dict(cond_nc=6, n_res_block=6, num_filters=[64, 128, 256]))
    g = AttentionLWBGenerator(cfg)
    sd = synth_state_dict(0)
    assert list(g.state_dict().keys()) == list(sd.keys())
    g.load_state_dict(sd, strict=True)
    # DDP-style "module." prefixes are stripped by the reference's loader before load_state_dict; strict=False works too
    g.load_state_dict({k: v for k, v in list(sd.items())[:10]}, strict=False)
    with pytest.raises(RuntimeError, match="CUDA"):
        g.forward_src(torch.zeros(1, 2, 6, 64, 64))


def test_weight_packing_layouts():
    from ipercore_b200 import ops
    w = torch.arange(2 * 3 * 3 * 3, dtype=torch.float32).reshape(2, 3, 3, 3)
    p = ops.pack_conv_weight(w, 2)
    assert p.w.shape == (2, 2, 27) and p.fmt == 2 and p.rows_total == 2 and p.K == 27
    # K order is (tap, cin): element (co=1, tap=4 (ky=1,kx=1), ci=2)
    # (the planes hold w * 2^k with max|w| * 2^k in [128, 256), undone exactly by the conv epilogue's w_scale_inv)
    assert 128.0 <= float(w.abs().max()) * p.scale < 256.0 and float(p.scale_inv) * p.scale == 1.0
    assert (float(p.w[0, 1, 4 * 3 + 2]) + float(p.w[1, 1, 4 * 3 + 2])) / p.scale == float(w[1, 2, 1, 1])
    wt = torch.randn(4, 5, 4, 4)
    pt = ops.pack_convT_weight(wt, 1)
    assert pt.w.shape == (1, 4 * 5, 4 * 4)
    # phase (py=1,px=0), tap (ta=0,tb=1): ky=0, kx=3
    torch.testing.assert_close(pt.w[0, 2 * 5 + 3, (0 * 2 + 1) * 4 + 2].float() / pt.scale, wt[2, 3, 0, 3], atol=2e-3, rtol=2e-3)
    hi_lo = ops.split_planes(torch.tensor([1.0001234, -3.14159265]), 2).float()
    torch.testing.assert_close(hi_lo.sum(0), torch.tensor([1.0001234, -3.14159265]), atol=1e-6, rtol=0)
    # format 3: e4m3 planes reproduce w and (w - fp16(w)) to ~2^-4 relative, with a power-of-two scale
    wr = (torch.rand(8, 64) - 0.5) * 0.2
    p3 = ops.PackedW(wr, 3)
    main, w_for_lo, wlo = p3.effective()
    assert p3.w8.dtype == torch.uint8 and p3.w8.shape == (8, 64) and abs(p3.cross_scale * 16384.0 * p3.sW - 1.0) < 1e-12
    assert float((w_for_lo - main).abs().max()) <= float(main.abs().max()) * 2 ** -4
    lo = wr - wr.half().float()
    assert float((wlo - lo).abs().max()) <= float(lo.abs().max()) * 2 ** -4 + 1e-12
    heads = ops.pack_heads_weight(torch.randn(3, 64, 5, 5), torch.randn(1, 64, 5, 5), 2)
    assert heads.w.shape == (2, 32, 320) and float(heads.w[:, 20:].abs().max()) == 0.0


def _staged_reference():
    from oracle import ref_runtime as rr
    return rr.ref_root() if rr.available() else None


@pytest.mark.skipif(_staged_reference() is None, reason="reference tree not staged (oracle/build_ref.py)")
def test_patch_install_against_reference():
    """install() wires the seams into the REAL iPERCore package (import level; runs in a subprocess to keep sys.modules clean)."""
    import subprocess
    import sys
    ref = _staged_reference()
    code = r"""
import sys, types
sys.path.insert(0, %r); sys.path.insert(0, %r)
import numpy as np; np.int = int; np.float = float
ed = types.ModuleType("easydict")
class AD(dict):
    def __getattr__(s, k):
        v = s[k]; return AD(v) if isinstance(v, dict) else v
ed.EasyDict = AD; sys.modules["easydict"] = ed
import ipercore_b200.patch as p
p.install()
import toml
from iPERCore.models.networks import NetworksFactory
cfg = AD(toml.load(%r)["Generator"])
g = NetworksFactory.get_by_name("AttLWB-SPADE", cfg=cfg, temporal=False)
assert type(g).__module__ == "ipercore_b200.generator" and len(g.state_dict()) == 221
from iPERCore.models import imitator as imod
from iPERCore.tools.human_digitalizer.renders import SMPLRenderer
assert SMPLRenderer.cal_bc_transform.__module__ == "ipercore_b200.patch"
assert imod.Imitator.inference.__module__ == "ipercore_b200.patch"
import neural_renderer
assert neural_renderer.__name__ == "ipercore_b200.neural_renderer"
print("OK")
""" % (ROOT, ref, os.path.join(ref, "assets", "configs", "neural_renders", "AttLWB-SPADE.toml"))
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and "OK" in out.stdout, out.stderr[-2000:]


def _halo_plan(mode, cin, rows, fuse_n=0):
    import numpy as np
    from ipercore_b200 import _lib
    buf = np.zeros(256, dtype=np.int32)
    n = _lib.lib.iper_conv_halo_plan(mode, cin, rows, fuse_n, buf.ctypes.data, buf.size)
    assert n > 0, _lib.lib.iper_last_error()
    n_loads, acc_blocks, box_rows = (int(v) for v in buf[:3])
    blk_phase = [int(v) for v in buf[3:7]]
    loads = buf[7:7 + 4 * n_loads].reshape(n_loads, 4)
    ne = int(loads[-1, 2] + loads[-1, 3])
    entries = buf[7 + 4 * n_loads:7 + 4 * n_loads + 13 * ne].reshape(ne, 13)
    assert n == 7 + 4 * n_loads + 13 * ne
    return acc_blocks, box_rows, loads, entries, blk_phase


def test_halo_tap_program_covers_every_tap_once():
    """Host logic of the halo kernel (conv_tc.cu build_halo_sched): every (phase, tap) of the layer appears exactly once,
    reads the view of the box that corresponds to its spatial offset, and the transposed conv's offsets agree with
    ConvTranspose2d(4, 2, 1) index algebra (out = 2*in - 1 + k) — in the per-(phase, tap) form and in the fused-N form."""
    from ipercore_b200._lib import IPER_CONV_ROW5, IPER_CONV_S1, IPER_CONVT_4S2
    cin, rows, tw = 128, 64, 16
    # 3x3 stride 1: tap (dy, dx) at K column (dy*3+dx)*Cin must read input offset (dy-1, dx-1)
    acc, box_rows, loads, ent, _ = _halo_plan(IPER_CONV_S1, cin, rows)
    assert acc == 1 and box_rows == (8 + 2) * tw and len(ent) == 9
    seen = set()
    for ox, oy, first, count in loads:
        for a_off, b_row, b_k, blk, nblk in ent[first:first + count, :5]:
            tap = b_k // cin
            dy, dx = divmod(tap, 3)
            assert b_k % cin == 0 and b_row == 0 and blk == 0 and nblk == 1
            assert a_off % tw == 0 and oy + a_off // tw == dy - 1 and ox == dx - 1
            seen.add(tap)
    assert seen == set(range(9))
    # heads: five vertical taps of one 32 x (4+4) box
    acc, box_rows, loads, ent, _ = _halo_plan(IPER_CONV_ROW5, 64, 32)
    assert acc == 1 and box_rows == 8 * 32 and len(loads) == 1 and tuple(loads[0][:2]) == (0, -2)
    assert [(int(e[0]) // 32, int(e[2]) // 64) for e in ent] == [(d, d) for d in range(5)]
    # transposed 4x4 s2 p1: output (2y+py, 2x+px) gathers input (y+oy, x+ox) through kernel index k = (2y+py) - 2(y+oy) + 1
    kidx = {0: (1, 3), 1: (0, 2)}          # pack_convT_weight: phase parity -> kernel indices of taps 0, 1

    def check(phase, tap, iy, ix):
        py, px, ta, tb = phase >> 1, phase & 1, tap >> 1, tap & 1
        assert kidx[py][ta] == py - 2 * iy + 1 and kidx[px][tb] == px - 2 * ix + 1

    acc, box_rows, loads, ent, blk_phase = _halo_plan(IPER_CONVT_4S2, cin, rows, fuse_n=0)
    assert acc == 4 and len(ent) == 16 and blk_phase == [0, 1, 2, 3]
    seen = set()
    for ox, oy, first, count in loads:
        for a_off, b_row, b_k, blk, nblk in ent[first:first + count, :5]:
            phase, tap = b_row // rows, b_k // cin
            assert b_row % rows == 0 and b_k % cin == 0 and blk == phase and nblk == 1
            check(phase, tap, oy + a_off // tw, ox)
            seen.add((phase, tap))
    assert len(seen) == 16
    # fused N: one entry per view and run of adjacent accumulator blocks; block b holds phase blk_phase[b]; CTA r of the
    # pair stages the whole weight boxes of blocks [acc + r*nblk/2, acc + (r+1)*nblk/2)
    acc, box_rows, loads, ent, blk_phase = _halo_plan(IPER_CONVT_4S2, cin, rows, fuse_n=1)
    assert acc == 4 and sorted(blk_phase) == [0, 1, 2, 3] and len(ent) == 11
    assert int(ent[0][4]) == 4 and int(ent[0][3]) == 0, "the first MMA group must initialise all four accumulator blocks"
    seen = []
    for ox, oy, first, count in loads:
        for e in ent[first:first + count]:
            a_off, b_row, b_k, blk, nblk = (int(v) for v in e[:5])
            fb_row, fb_k = e[5:9].reshape(2, 2), e[9:13].reshape(2, 2)
            assert nblk in (1, 2, 4) and blk + nblk <= 4 and blk % nblk == 0
            iy = oy + a_off // tw
            if nblk == 1:
                assert b_row // rows == blk_phase[blk]
                check(b_row // rows, b_k // cin, iy, ox)
                seen.append((b_row // rows, b_k // cin))
            else:
                for r in range(2):
                    for i in range(nblk // 2):
                        b = blk + r * (nblk // 2) + i
                        phase, tap = int(fb_row[r][i]) // rows, int(fb_k[r][i]) // cin
                        assert phase == blk_phase[b]
                        check(phase, tap, iy, ox)
                        seen.append((phase, tap))
    assert len(seen) == 16 and len(set(seen)) == 16
