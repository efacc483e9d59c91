"""The zero-edit integration route on a GPU with the REAL reference classes (VERDICT r01 item 2 / SURVEY.md §8b seam B4):

    ipercore_b200.patch.install()  ->  iPERCore.models.imitator.Imitator(opt).source_setup(...) / .inference(...)

against the stock reference (same classes, torch true fp32, rasteriser = host C oracle) on the same inputs: same
pred_%08d.png files within one code value, same source-side uv image / background / face maps.  The stock run is stored in
tests/golden/imitator_S*.npz (make_golden.py imitator: face maps in full, f2pts as a SHA-256, a fixed seeded sample of the
pixels of the uv image, the background and every frame).  The patched run needs the reference's own Python classes, staged
under oracle/_ref by oracle/build_ref.py; SMPLH pkl and checkpoint are synthetic files in the reference's formats.  The
patched arm runs in its own process because install() patches classes process-wide.
"""
import hashlib
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))


def _run(patched, work, size, frames, batch, temporal=0):
    cmd = [sys.executable, os.path.join(ROOT, "tests", "ref_run_imitator.py"), "--patched", str(patched), "--work", work,
           "--size", str(size), "--frames", str(frames), "--batch", str(batch), "--temporal", str(temporal)]
    p = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=1500)
    assert p.returncode == 0, p.stdout[-4000:]
    d = os.path.join(work, "patched" if patched else "stock")
    return d, json.load(open(os.path.join(d, "run.json")))


@pytest.mark.parametrize("temporal", [0, 1])
def test_real_imitator_patched_equals_stock(temporal, tmp_path, golden_dir):
    """temporal=0: the batched engine replaces Imitator.inference; temporal=1: the upstream bs=1 loop with its TemporalFIFO
    recurrence (imitator.py:18-127, 341-380) drives the B200 generator / renderer frame by frame."""
    from oracle import ref_runtime as rr
    if not rr.available():
        pytest.skip("reference tree not staged (oracle/build_ref.py)")
    import cv2
    import make_golden
    S, T, B, _ = make_golden.IMITATOR_CASES[temporal]
    g = np.load(os.path.join(golden_dir, make_golden.imitator_golden_name(S, temporal)))
    meta = json.loads(str(g["meta"]))
    d1, r1 = _run(1, str(tmp_path), S, T, B, temporal)
    assert meta["generator"].startswith("iPERCore.") and meta["nr_is_stub"]
    assert r1["generator"] == "ipercore_b200.generator" and r1["renderer_nr"] == "ipercore_b200.neural_renderer"
    assert meta["outputs"] == r1["outputs"] == ["pred_%08d.png" % i for i in range(T)]
    s1 = np.load(os.path.join(d1, "source.npz"))
    np.testing.assert_array_equal(s1["fim"], g["fim"])                        # source face-index maps bit-exact
    assert hashlib.sha256(np.ascontiguousarray(s1["f2pts"], np.float32).tobytes()).hexdigest() == str(g["f2pts_sha256"])
    uv_px = g["uv_px"]
    np.testing.assert_allclose(s1["uv_img"].reshape(3, S * S)[:, uv_px], g["uv_img"], atol=1e-5, rtol=0)
    np.testing.assert_allclose(s1["bg"].reshape(3, S * S)[:, uv_px], g["bg"], atol=1e-3, rtol=0)   # forward_bg on the tensor path
    worst, frac = 0, 0.0
    for k, name in enumerate(r1["outputs"]):
        b = cv2.imread(os.path.join(d1, name), cv2.IMREAD_COLOR)
        assert b.shape == (S, S, 3)
        d = np.abs(b.reshape(S * S, 3)[g["px"]].astype(np.int32) - g["frames"][k].astype(np.int32))
        worst, frac = max(worst, int(d.max())), max(frac, float((d > 0).mean()))
    print("real Imitator, patched vs stock (%s): max code diff %d, worst fraction of differing sampled pixels %.4f; "
          "patched %.2fs + %.2fs (source_setup + inference)" % (meta["device"], worst, frac, r1["source_setup_s"],
                                                                 r1["inference_s"]))
    assert worst <= 1 and frac < 0.02
