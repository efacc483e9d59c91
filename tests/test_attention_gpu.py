"""iper_warp_attention (ops.cu) against a float64 restatement of the reference's SelfAttentionLWB
(attlwb_spade_resunet.py:208-252): warp every source with F.grid_sample(align_corners=False, zeros), project it with
fk / fv, project the target with fq, softmax over sources of K.q / sqrt(C), sum of the weighted values.  The kernel
computes the same thing with the projections hoisted to the source side (ops.attention_source_weight), so this also
checks that algebra, including the Wk^T bq column.

Every case runs on the schedule the process starts with (the chunked kernel unless IPER_ATT_WIDE is set).  The library
reads IPER_ATT_WIDE once per process, so the pixel-per-warp schedules run in child processes (run_variant), one per
setting, which also record the names of the kernels they launched."""
import json
import math
import os
import re
import subprocess
import sys
from typing import NamedTuple

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
SENTINEL16 = 0x7E5A          # an fp16 NaN; as bytes 0x5A 0x7E in the e4m3 planes of format 3


# ----------------------------------------------------------------------------------------------------------------------
# child processes for the process-wide switches
# ----------------------------------------------------------------------------------------------------------------------
_CHILD = r"""
import json, os, sys
d, module, func, keys = sys.argv[1], sys.argv[2], sys.argv[3], sys.argv[4:]
sys.path[:0] = [os.getcwd(), os.path.join(os.getcwd(), "tests")]
import importlib
import numpy as np
helpers = importlib.import_module("test_attention_gpu")
fn = getattr(importlib.import_module(module), func)
inputs = dict(np.load(os.path.join(d, "in.npz")))
out, names = helpers.profiled_kernels(lambda: fn(inputs), os.path.join(d, "trace.json"))
np.savez(os.path.join(d, "out.npz"), **out)
with open(os.path.join(d, "child.json"), "w") as f:
    json.dump(dict(kernels=names, env={k: os.environ.get(k) for k in keys}), f)
"""


def profiled_kernels(fn, trace_path):
    """(fn(), sorted names of the CUDA kernels it launched), from a torch.profiler trace written to trace_path."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    prof.export_chrome_trace(trace_path)
    with open(trace_path) as f:
        events = json.load(f)["traceEvents"]
    return out, sorted({e["name"] for e in events if e.get("cat") == "kernel"})


def run_variant(tmp_path, env, module, func, inputs, timeout=900):
    """Run module.func(inputs) -> dict of arrays in a fresh interpreter whose environment is ours updated with `env`
    (a value None removes the variable).  Inputs and outputs travel as .npz under tmp_path.  Returns (outputs, names of
    the CUDA kernels the call launched); asserts that the child saw `env`."""
    tag = "_".join("%s-%s" % (k, v) for k, v in sorted(env.items()))
    d = tmp_path / ("child_" + tag)
    d.mkdir()
    np.savez(d / "in.npz", **inputs)
    child_env = {k: v for k, v in os.environ.items() if k not in env}
    child_env.update({k: v for k, v in env.items() if v is not None})
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + ["-c", _CHILD, str(d), module, func] + list(env)
    r = subprocess.run(cmd, cwd=ROOT, env=child_env, capture_output=True, text=True, timeout=timeout)
    assert r.returncode == 0, "child %s failed:\n%s\n%s" % (tag, r.stdout[-4000:], r.stderr[-4000:])
    with open(d / "child.json") as f:
        info = json.load(f)
    assert info["env"] == env, "child environment %s, wanted %s" % (info["env"], env)
    with np.load(d / "out.npz") as z:
        out = {k: z[k] for k in z.files}
    return out, info["kernels"]


# ----------------------------------------------------------------------------------------------------------------------
# inputs
# ----------------------------------------------------------------------------------------------------------------------
def _rand(shape, seed, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    return (torch.rand(shape, generator=g) * 2 - 1) * scale


class Case(NamedTuple):
    C: int
    ns: int
    flow: str
    B: int
    h: int
    w: int
    p_in: int          # planes format of the target features
    p_out: int         # planes format of the output
    window: bool       # xt and out as channel windows of wider buffers
    seed: int

    def __str__(self):
        return "C%d-ns%d-%s-%dx%dx%d-P%d%d%s" % (self.C, self.ns, self.flow, self.B, self.h, self.w, self.p_in, self.p_out,
                                                 "-win" if self.window else "")


FLOWS = ("realframe", "uniform", "background", "border", "nonfinite")
# (xt, out) formats att_block produces for precision fp16, fp16x2, fp16f8, mixed
FORMATS = ((1, 1), (2, 2), (3, 3), (2, 1))
# B*h*w is not a multiple of any chunk size (32 / 16 / 8 pixels for C = 64 / 128 / 256): every chunk walk ends in a tail
SHAPES = ((3, 5, 7), (2, 13, 10), (1, 9, 20))


def _cases():
    out = []
    for ic, C in enumerate((64, 128, 256)):
        for i_ns, ns in enumerate((1, 2, 3, 4, 5, 8)):
            for i_f, flow in enumerate(FLOWS):
                B, h, w = (2, 37, 29) if flow == "realframe" else SHAPES[(i_ns + 2 * i_f + ic) % 3]
                p_in, p_out = FORMATS[(i_ns + i_f) % 4]
                out.append(Case(C, ns, flow, B, h, w, p_in, p_out, (i_ns + i_f + ic) % 2 == 0, 1000 + len(out)))
    return out


CASES = _cases()
# more pixels than one grid-stride trip of the chunked kernel covers (1776 CTAs x 8 warps x chunk)
LARGE = [Case(256, 5, "realframe", 8, 128, 128, 2, 2, False, 7001), Case(128, 3, "realframe", 4, 256, 256, 3, 3, True, 7002),
         Case(64, 2, "realframe", 8, 256, 256, 2, 1, True, 7003)]


def _coords(n, shape, g):
    """border-tap coordinates along an axis of n pixels: pixel centres, +-1, half a pixel outside, arbitrary"""
    centres = (2 * torch.randint(0, n, shape, generator=g).float() + 1) / n - 1
    choice = torch.randint(0, 6, shape, generator=g)
    anywhere = torch.rand(shape, generator=g) * 2 - 1
    vals = torch.stack([centres, torch.full(shape, -1.0), torch.full(shape, 1.0), torch.full(shape, -1 - 1.0 / n),
                        torch.full(shape, 1 + 1.0 / n), anywhere], -1)
    return vals.gather(-1, choice[..., None])[..., 0]


def _flow(case):
    B, ns, h, w = case.B, case.ns, case.h, case.w
    g = torch.Generator().manual_seed(case.seed + 1)
    if case.flow == "uniform":
        return (torch.rand((B, ns, h, w, 2), generator=g) * 2 - 1) * 1.3
    if case.flow == "background":
        return torch.full((B, ns, h, w, 2), -2.0)
    if case.flow == "border":
        return torch.stack([_coords(w, (B, ns, h, w), g), _coords(h, (B, ns, h, w), g)], -1)
    if case.flow == "nonfinite":
        T = (torch.rand((B, ns, h, w, 2), generator=g) * 2 - 1) * 1.1
        bad = torch.tensor([float("nan"), float("inf"), -float("inf"), 1e30, -1e30])
        hit = torch.rand((B, ns, h, w, 2), generator=g) < 0.15
        T = torch.where(hit, bad[torch.randint(0, 5, (B, ns, h, w, 2), generator=g)], T)
        T[:, :, 0, 0] = float("nan")             # one pixel where no source is usable
        return T
    # real-frame-like: Tst's background value -2 outside the body, a smooth in-range field inside one blob per source
    ys, xs = torch.meshgrid(torch.arange(h).float(), torch.arange(w).float(), indexing="ij")
    T = torch.full((B, ns, h, w, 2), -2.0)
    r = math.sqrt(0.15 * h * w / math.pi)
    for b in range(B):
        for s in range(ns):
            cy, cx = (torch.rand(2, generator=g) * 0.6 + 0.2) * torch.tensor([h, w])
            a = torch.rand(4, generator=g)
            inside = (ys - cy) ** 2 + (xs - cx) ** 2 <= r * r
            gx = ((2 * xs + 1) / w - 1) * 0.8 + 0.1 * torch.sin(ys * (0.2 + a[0]) + 6 * a[1])
            gy = ((2 * ys + 1) / h - 1) * 0.8 + 0.1 * torch.cos(xs * (0.2 + a[2]) + 6 * a[3])
            T[b, s, ..., 0] = torch.where(inside, gx, -2.0)
            T[b, s, ..., 1] = torch.where(inside, gy, -2.0)
    return T


def _problem(case):
    """seeded float32 inputs (CPU) drawn as test_stem_and_attention_kernels did, bq != 0 so the k0 column matters"""
    C, ns, s = case.C, case.ns, case.seed * 16
    return dict(src=_rand((ns, C, case.h, case.w), s + 1), xt=_rand((case.B, C, case.h, case.w), s + 2),
                wq=_rand((C, C, 1, 1), s + 3, 0.1), bq=_rand((C,), s + 4, 0.3), wk=_rand((C, C, 1, 1), s + 5, 0.2),
                bk=_rand((C,), s + 6, 0.3), wv=_rand((C, C, 1, 1), s + 7, 0.2), bv=_rand((C,), s + 8, 0.1), T=_flow(case))


def _windows(case):
    """(xt pitch, xt coff, out pitch, out coff)"""
    C = case.C
    return (C + 24, 16, C + 16, 8) if case.window else (C, 0, C, 0)


def _device_inputs(case, pr, dev):
    """xt Planes (possibly a window of a wider buffer holding other features), kv, bias_v, T on `dev`"""
    from ipercore_b200 import ops
    from ipercore_b200.ops import Planes
    xp, xo, _, _ = _windows(case)
    wide = torch.cat([_rand((case.B, xo, case.h, case.w), case.seed * 16 + 9), pr["xt"],
                      _rand((case.B, xp - xo - case.C, case.h, case.w), case.seed * 16 + 10)], 1)
    xt = Planes.from_nchw(wide.to(dev), case.p_in).window(xo, case.C)
    wsrc = ops.attention_source_weight(pr["wq"], pr["bq"], pr["wk"], pr["wv"])          # fp32, as the generator packs it
    src = pr["src"].to(dev)
    kv = torch.einsum("oc,schw->shwo", wsrc.to(dev)[:, :, 0, 0].double(), src.double()).float().contiguous()
    return xt, kv, pr["bv"].to(dev), pr["T"].to(dev).contiguous()


def _empty_out(case, dev):
    from ipercore_b200.ops import Planes
    _, _, op, oo = _windows(case)
    buf = Planes.empty(case.p_out, case.B, case.h, case.w, case.C, dev, pitch=op)
    buf.data.view(torch.int16).fill_(SENTINEL16)
    return buf, buf.window(oo, case.C)


def _raw_planes(p):
    """every stored plane of a Planes buffer as an integer tensor (N, H, W, pitch)"""
    d = p.data
    if p.P == 1:
        return [d[0].view(torch.int16)]
    if p.P == 2:
        return [d[0].view(torch.int16), d[1].view(torch.int16)]
    return [d[0].view(torch.int16)] + list(d[1].reshape(-1).view(torch.uint8).reshape(2, p.N, p.H, p.W, p.pitch))


# ----------------------------------------------------------------------------------------------------------------------
# reference and checks
# ----------------------------------------------------------------------------------------------------------------------
def reference(pr, xq, dev):
    """float64 SelfAttentionLWB of the stored target values xq (B,C,h,w).  A flow the kernel treats as 'every tap out of
    range' (non-finite, or far outside the map) is replaced by the background value -2 first: that source then
    contributes K = bk, V = bv, which is what the kernel's bilinear_taps contract gives."""
    d = lambda t: t.to(dev, torch.float64)
    src, T = d(pr["src"]), d(pr["T"])
    bad = (~torch.isfinite(T) | (T.abs() >= 1e20)).any(-1, keepdim=True)
    T = torch.where(bad, torch.full_like(T, -2.0), T)
    Wq, Wk, Wv = (d(pr[k])[:, :, 0, 0] for k in ("wq", "wk", "wv"))
    bq, bk, bv = (d(pr[k])[:, None, None] for k in ("bq", "bk", "bv"))
    C = src.shape[1]
    out = []
    for b in range(T.shape[0]):
        warp = F.grid_sample(src, T[b], mode="bilinear", padding_mode="zeros", align_corners=False)    # (ns,C,h,w)
        K = torch.einsum("oc,schw->sohw", Wk, warp) + bk
        V = torch.einsum("oc,schw->sohw", Wv, warp) + bv
        q = torch.einsum("oc,chw->ohw", Wq, d(xq[b])) + bq
        logit = (K * q).sum(1, keepdim=True) / math.sqrt(C)
        out.append((torch.softmax(logit, 0) * V).sum(0))
    return torch.stack(out)


def format_unit(a, P):
    """one unit of planes format P at magnitude a: fp16 spacing (P=1), that of the fp16 lo plane (P=2) or of the e4m3 lo
    plane (P=3, 3 mantissa bits of a remainder of at most half an fp16 step)"""
    e = torch.frexp(a.float().clamp_min(2.0 ** -14)).exponent
    ulp16 = torch.ldexp(torch.ones_like(a, dtype=torch.float32), e - 11)
    if P == 1:
        return ulp16
    if P == 2:
        return torch.clamp_min(ulp16 * 2.0 ** -11, 2.0 ** -24)
    return torch.clamp_min(ulp16 * 2.0 ** -4, 2.0 ** -23)


def check_output(out, exp, atol, label):
    """out (a Planes window) against the fp64 result rounded through out's format: atol + one unit of that format"""
    from ipercore_b200.ops import Planes
    exp_r = Planes.from_nchw(exp.float().to(out.data.device), out.P).to_nchw()
    got = out.to_nchw()
    assert torch.isfinite(got).all(), "%s: non-finite output (an unwritten pixel reads back as the NaN sentinel)" % label
    err = (got - exp_r).abs()
    tol = atol + format_unit(exp_r.abs(), out.P)
    print("%-44s max |err| %.2e (%.2f of the bound)" % (label, float(err.max()), float((err / tol).max())))
    assert (err <= tol).all(), "%s: max err %.3e at %s" % (label, float(err.max()), (err / tol).argmax())
    if out.P == 3:      # the a8 plane (e4m3(8 x), fed to the fp8 cross-term MMAs) must hold the same value
        a8 = _raw_planes(out)[1][..., out.coff:out.coff + out.C].view(torch.float8_e4m3fn).float() / 8.0
        v = got.permute(0, 2, 3, 1)
        assert ((a8 - v).abs() <= v.abs() * 0.07 + 2.0 ** -12).all(), "%s: a8 plane disagrees" % label


def check_outside_kept(buf, before, coff, C, label):
    """channels of buf outside [coff, coff+C) still hold their sentinel bits, in every plane"""
    keep = torch.ones(buf.pitch, dtype=torch.bool, device=buf.data.device)
    keep[coff:coff + C] = False
    for i, (a, b) in enumerate(zip(_raw_planes(buf), before)):
        assert torch.equal(a[..., keep], b[..., keep]), "%s: plane %d written outside the channel window" % (label, i)


def _run(case, dev, pr=None):
    """(problem, stored target values, output buffer, output window) after one iper_warp_attention call"""
    from ipercore_b200 import ops
    pr = pr or _problem(case)
    xt, kv, bv, T = _device_inputs(case, pr, dev)
    buf, out = _empty_out(case, dev)
    before = [t.clone() for t in _raw_planes(buf)]
    ops.warp_attention(xt, kv, bv, T, out)
    torch.cuda.synchronize()
    check_outside_kept(buf, before, out.coff, case.C, str(case))
    return pr, xt.to_nchw(), buf, out


@pytest.mark.parametrize("case", CASES, ids=str)
def test_warp_attention_matches_fp64(case):
    pr, xq, _, out = _run(case, DEV)
    exp = reference(pr, xq.cpu(), "cpu")
    if case.flow == "background":    # no tap of any source lands in a map: softmax of equal logits of the value bias_v
        assert float((exp - pr["bv"].double()[None, :, None, None]).abs().max()) < 1e-12
    check_output(out, exp, 1e-6 if case.flow == "background" else 3e-5, str(case))


@pytest.mark.parametrize("case", LARGE, ids=str)
def test_warp_attention_large_maps(case):
    """several grid-stride trips of every warp; reference in float64 on the GPU"""
    pr, xq, _, out = _run(case, DEV)
    check_output(out, reference(pr, xq, DEV), 3e-5, str(case))


# ----------------------------------------------------------------------------------------------------------------------
# schedules: IPER_ATT_WIDE unset (chunked), 0, 1, 2 (pixel-per-warp)
# ----------------------------------------------------------------------------------------------------------------------
# every (C, NSMAX) instantiation, each bucket both full and partly used, with background, border taps and bad flows
SUBSET = [c for c in CASES if c.flow in ("realframe", "border", "nonfinite")]
SCHEDULES = (None, "0", "1", "2")


def _schedule(v):
    """the schedule iper_warp_attention picks for IPER_ATT_WIDE = v (atoi semantics, unset = chunked)"""
    if v is None:
        return "chunk"
    try:
        w = int(v)
    except ValueError:
        w = 0
    return "chunk" if w == 3 else "W%d" % (w if w in (1, 2) else 0)


def _pack_subset():
    arrays = {}
    for i, case in enumerate(SUBSET):
        pr = _problem(case)
        xt, kv, bv, T = _device_inputs(case, pr, DEV)
        arrays.update({"c%d_xt" % i: xt.data.cpu().numpy(), "c%d_kv" % i: kv.cpu().numpy(), "c%d_bv" % i: bv.cpu().numpy(),
                       "c%d_T" % i: T.cpu().numpy(), "c%d_meta" % i: np.array([xt.P, xt.coff, xt.C])})
    return arrays


def child_attention(inputs):
    """every SUBSET case through iper_warp_attention on this process's schedule -> raw output buffers"""
    from ipercore_b200 import ops
    from ipercore_b200.ops import Planes
    out = {}
    for i, case in enumerate(SUBSET):
        P, coff, C = (int(v) for v in inputs["c%d_meta" % i])
        xt = Planes(torch.from_numpy(inputs["c%d_xt" % i]).to(DEV), fmt=P).window(coff, C)
        buf, o = _empty_out(case, DEV)
        t = lambda k: torch.from_numpy(inputs["c%d_%s" % (i, k)]).to(DEV)
        ops.warp_attention(xt, t("kv"), t("bv"), t("T"), o)
        out["c%d_out" % i] = buf.data.cpu().numpy()
    torch.cuda.synchronize()
    return out


def _attention_kernels(names):
    """(kind, C, NSMAX, WIDE or None) of every warp-attention kernel in a list of demangled kernel names"""
    out = set()
    for n in names:
        m = re.search(r"warp_attention_chunk_kernel<(\d+), (\d+)>", n)
        if m:
            out.add(("chunk", int(m[1]), int(m[2]), None))
        m = re.search(r"warp_attention_kernel<(\d+), (\d+), (\d+)>", n)
        if m:
            out.add(("W%s" % m[3], int(m[1]), int(m[2]), int(m[3])))
    return out


def test_schedules_agree_and_launch_their_kernels(tmp_path):
    """The four schedules use the same arithmetic order per pixel, so their outputs are compared bit for bit; where they
    are not bitwise equal, within 1e-6 relative plus one unit of the output format (reported).  Each run's profiler
    trace names the kernels it launched: one per (C, NSMAX) instantiation, of its own schedule only."""
    from ipercore_b200.ops import Planes
    inputs = _pack_subset()
    here = os.environ.get("IPER_ATT_WIDE")
    outs, kernels = {}, {}
    outs[here], kernels[here] = profiled_kernels(lambda: child_attention(inputs), str(tmp_path / "trace_inprocess.json"))
    for v in SCHEDULES:
        if _schedule(v) != _schedule(here):
            outs[v], kernels[v] = run_variant(tmp_path, {"IPER_ATT_WIDE": v}, "test_attention_gpu", "child_attention", inputs)
    by_sched = {_schedule(v): v for v in outs}
    assert sorted(by_sched) == ["W0", "W1", "W2", "chunk"]
    want = {(c.C, 2 if c.ns <= 2 else (4 if c.ns <= 4 else 8)) for c in SUBSET}
    for sched, v in sorted(by_sched.items()):
        att = _attention_kernels(kernels[v])
        print("schedule %-5s (IPER_ATT_WIDE=%s) ran: %s" % (sched, v, ", ".join(sorted({re.sub(r"\(.*", "", n)
                                                                                       for n in kernels[v] if "warp_attention" in n}))))
        assert {k[0] for k in att} == {sched}, (sched, att)
        assert {(k[1], k[2]) for k in att} == want, (sched, sorted(att), sorted(want))
    base = outs[by_sched["chunk"]]
    for sched in ("W0", "W1", "W2"):
        o = outs[by_sched[sched]]
        same, worst = 0, 0.0
        for i, case in enumerate(SUBSET):
            a, b = base["c%d_out" % i], o["c%d_out" % i]
            if np.array_equal(a.view(np.uint16), b.view(np.uint16)):
                same += 1
                continue
            oo = _windows(case)[3]
            va = Planes(torch.from_numpy(a).to(DEV), C=case.C, coff=oo, fmt=case.p_out).to_nchw()
            vb = Planes(torch.from_numpy(b).to(DEV), C=case.C, coff=oo, fmt=case.p_out).to_nchw()
            d = (va - vb).abs()
            worst = max(worst, float((d / va.abs().clamp_min(1e-30)).max()))
            assert (d <= 1e-6 * va.abs() + format_unit(va.abs(), case.p_out)).all(), \
                "%s: schedule %s differs from the chunked one by %.2e" % (case, sched, float(d.max()))
        print("schedule %s vs chunk: %d of %d cases bitwise equal; max relative difference of the others %.2e"
              % (sched, same, len(SUBSET), worst))
