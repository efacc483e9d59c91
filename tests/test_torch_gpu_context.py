"""Context measurement (not a parity test): the plain PyTorch/cuDNN formulation of the per-frame path on the same B200 —
"the existing Blackwell kernel to beat" of SURVEY.md §8d / BASELINE.md §3 — using the oracle's torch-functional
restatement moved to cuda:0.  Prints the rates (and writes them to torch_gpu_baseline.json in the test's temporary
directory); asserts only sanity."""
import json
import os
import time

import numpy as np
import pytest
import torch

from oracle import generator_ref, synth, weights

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("S", [512])
def test_pytorch_cudnn_path_timing(S, template, tmp_path):
    import make_golden
    dev = "cuda:0"
    sd = {k: v.to(dev) for k, v in weights.synth_state_dict(0).items()}
    inp = {k: torch.from_numpy(v).to(dev) for k, v in make_golden.gen_inputs(S).items()}
    res = {}
    for name, tf32, autocast in (("fp32_tf32_default", True, None), ("fp32_ieee", False, None),
                                 ("bf16_autocast", True, torch.bfloat16), ("fp16_autocast", True, torch.float16)):
        torch.backends.cudnn.allow_tf32 = tf32
        torch.backends.cuda.matmul.allow_tf32 = tf32
        with torch.no_grad(), torch.autocast("cuda", dtype=autocast, enabled=autocast is not None):
            se, sr = generator_ref.forward_src(sd, inp["src_inputs"])
            for bs in (1, 16):
                x = inp["tsf_inputs"].repeat(bs, 1, 1, 1); T = inp["Tst"].repeat(bs, 1, 1, 1, 1)
                se_b = [f.repeat(bs, 1, 1, 1) for f in se]; sr_b = [f.repeat(bs, 1, 1, 1) for f in sr]
                for _ in range(3):
                    generator_ref.forward_tsf(sd, x, se_b, sr_b, T)
                torch.cuda.synchronize()
                n = 20 if bs == 1 else 4
                t0 = time.perf_counter()
                for _ in range(n):
                    img, mask = generator_ref.forward_tsf(sd, x, se_b, sr_b, T)
                torch.cuda.synchronize()
                res["%s_bs%d_fps" % (name, bs)] = n * bs / (time.perf_counter() - t0)
    torch.backends.cudnn.allow_tf32 = True
    print("PyTorch/cuDNN forward_tsf %dx%d on %s:" % (S, S, torch.cuda.get_device_name(0)), json.dumps(res))
    json.dump(res, open(os.path.join(tmp_path, "torch_gpu_baseline.json"), "w"), indent=1)
    assert all(v > 0 for v in res.values())
