"""Helper process of tests/test_reference_integration_gpu.py: run the REAL iPERCore Imitator (staged reference tree,
oracle/ref_runtime.py) — source_setup + inference — either stock (reference modules on torch/cuDNN in true fp32, the
rasteriser stubbed by the host C oracle) or with ``ipercore_b200.patch.install()`` applied first (zero-edit route of
INTEGRATION.md §2), and leave pred_*.png + a small json behind.

    python tests/ref_run_imitator.py --patched {0,1} --work DIR --size S --frames T [--batch B] [--device cuda:0]
"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--patched", type=int, required=True)
    ap.add_argument("--work", required=True)
    ap.add_argument("--size", type=int, default=256)
    ap.add_argument("--frames", type=int, default=5)
    ap.add_argument("--batch", type=int, default=2)
    ap.add_argument("--device", default="cuda:0")
    ap.add_argument("--ns", type=int, default=2)
    ap.add_argument("--temporal", type=int, default=0)
    a = ap.parse_args()
    import numpy as np
    import torch
    from oracle import ref_runtime as rr
    torch.backends.cudnn.allow_tf32 = False           # the stock arm is the fp32 reference, not its TF32 approximation
    torch.backends.cuda.matmul.allow_tf32 = False
    rr.install_import_shims(stub_renderer=not a.patched)
    if a.patched:
        import ipercore_b200.patch as b200
        b200.install(precision="fp16x2", batch=a.batch)           # BEFORE iPERCore.models is imported
    opt, model = rr.make_opt(a.work, image_size=a.size, num_source=a.ns)
    opt.temporal = bool(a.temporal)           # deploy.toml:40; true = TemporalFIFO recurrence through the upstream bs=1 loop
    out_dir = os.path.join(a.work, "patched" if a.patched else "stock")
    os.makedirs(out_dir, exist_ok=True)
    im = rr.build_imitator(opt, a.device)
    sync = torch.cuda.synchronize if a.device.startswith("cuda") else (lambda: None)
    src_smpl, tgt = rr.synthetic_clip(model, a.frames, ns=a.ns)
    paths = rr.write_source_images(a.work, a.ns, a.size)
    t0 = time.time()
    info = im.source_setup(paths, src_smpl, masks=None, bg_img=None, offsets=0, links_ids=None)
    sync()
    t1 = time.time()
    outs = im.inference(tgt, cam_strategy="smooth", output_dir=out_dir, prefix="pred_", verbose=False)
    sync()
    t2 = time.time()
    np.savez_compressed(os.path.join(out_dir, "source.npz"), uv_img=info["uv_img"].float().cpu().numpy(),
                        bg=info["bg"].float().cpu().numpy(), f2pts=info["f2pts"].float().cpu().numpy(),
                        fim=info["fim"].cpu().numpy())
    json.dump(dict(generator=type(im.generator).__module__, renderer_nr=sys.modules["neural_renderer"].__name__,
                   nr_is_stub=bool(getattr(sys.modules["neural_renderer"], "IS_ORACLE_STUB", False)),
                   source_setup_s=t1 - t0, inference_s=t2 - t1, outputs=[os.path.basename(p) for p in outs]),
              open(os.path.join(out_dir, "run.json"), "w"))


if __name__ == "__main__":
    main()
