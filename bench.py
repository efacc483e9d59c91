#!/usr/bin/env python
"""bench.py — 512x512 motion-imitation frames/sec (BASELINE.json metric) on N B200s of one node.

    python bench.py --gpus 1 --steps 3 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...      # the reference's algorithm on the host cores (oracle port), rank 0 only

Workload (BASELINE.json configs[1], SURVEY.md §8d config 2): one source set (ns=2) -> 300 synthetic target SMPL poses at
512x512 per GPU; a "step" is one pass of the per-frame hot path (rows a1-a15) over those 300 frames in batches of B.
`value`  : frames/s with the 300 frames' vertices/cameras already resident in HBM (whole job, all ranks; weak scaling:
           every rank synthesizes its own 300-frame clip, no collective on the data path).
`e2e`    : the same through the public host API FrameEngine.synthesize(): pinned host vertices in, uint8 frames out,
           H2D/D2H inside the timed region.
`roofline`: conv stack (tcgen05 implicit GEMM) — algorithmic 285.93 GFLOP/frame (SURVEY.md §8a) over the summed CUDA-event
           duration of the conv launches of one batch, against the measured bf16 GEMM peak in MEASURED_PEAKS.json.
`cpu_baseline`: oracle port of the reference path (CPU restatement, torch fp32 on all host cores), bounded sample.
Weights are synthetic (oracle/weights.py; the real checkpoint is not available offline), data synthetic.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "tests", "golden")):
    if p not in sys.path:
        sys.path.insert(0, p)

CFG = dict(name="AttLWB-SPADE", BGNet=dict(cond_nc=4, n_res_block=6, num_filters=[64, 128, 128, 256]),
           SIDNet=dict(cond_nc=6, n_res_block=6, num_filters=[64, 128, 256]),
           TSFNet=dict(cond_nc=6, n_res_block=6, num_filters=[64, 128, 256]))
FLOPS_PER_FRAME_512 = 285.93e9          # SURVEY.md §8a, 76 convs of forward_tsf, ns=2


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="imitate", choices=["imitate", "train"],
                    help="imitate = BASELINE.json configs[1] (the headline); train = configs[4], one G + D + VGG training step per rank")
    ap.add_argument("--size", type=int, default=512)
    ap.add_argument("--frames", type=int, default=300)
    ap.add_argument("--batch", type=int, default=60)
    ap.add_argument("--ns", type=int, default=2)
    ap.add_argument("--precision", default="fp16x2", choices=["fp16x2", "fp16", "fp16f8", "mixed"])
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--streams", type=int, default=1, help="engines replaying alternate batches on separate streams")
    ap.add_argument("--dump-layers", default="", help="write the per-launch conv timing table (JSON) to this path")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-frames", type=int, default=8)
    ap.add_argument("--profile-batch", action="store_true",
                    help="for ncu --profile-from-start off: warm up, then run exactly ONE eager batch between cudaProfilerStart/Stop and exit")
    ap.add_argument("--no-parity", action="store_true", help="skip the oracle check of sampled frames of the last step")
    ap.add_argument("--no-lib-baseline", action="store_true", help="skip the reference-generator-on-cuDNN side leg")
    ap.add_argument("--no-png", action="store_true", help="skip the e2e pass that also writes the PNG files")
    ap.add_argument("--no-strong", action="store_true", help="N>1: skip the strong-scaling pass (one clip split over ranks)")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write what the last timed step computed to DIR/<name>.npy (float32/float64, <= 64 MB in all), "
                         "so two builds can be compared output for output")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    return args


DUMP_BUDGET = 64 * 10 ** 6 - 2 ** 16       # bytes of .npy files --dump-outputs may write (room left for the headers)


def dump_frames(out_dir, frames_d):
    """uint8 BGR frames (T,S,S,3) of the last timed step -> out_dir/frames.npy (float32, codes 0..255) and
    out_dir/frame_ids.npy (float64 clip indices).  A clip larger than the budget is cut to a fixed seeded sample of
    whole frames, the same sample for the same arguments."""
    import numpy as np
    import torch
    T = frames_d.shape[0]
    n = max(1, min(T, (DUMP_BUDGET - 8 * T) // (frames_d[0].numel() * 4)))
    ids = np.arange(T) if n == T else np.sort(np.random.Generator(np.random.PCG64(0)).choice(T, n, replace=False))
    frames = frames_d[torch.as_tensor(ids, device=frames_d.device)].float().cpu().numpy()
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "frames.npy"), frames)
    np.save(os.path.join(out_dir, "frame_ids.npy"), ids.astype(np.float64))


# ----------------------------------------------------------------------------------------------------------------------
# synthetic workload (oracle.synth only GENERATES inputs here)
# ----------------------------------------------------------------------------------------------------------------------
def make_workload(args, rank):
    import numpy as np
    from oracle import synth
    tpl = synth.load_template()
    S, ns = args.size, args.ns
    cams, verts = synth.pose_sweep(tpl, args.frames, total=300, start=rank * args.frames)
    scams, sverts = synth.source_views(tpl, ns)
    return dict(tpl=tpl, cams=cams, verts=verts, scams=scams, sverts=sverts,
                src_img=synth.smooth_image((ns, 3, S, S), seed=1), uv_img=synth.smooth_image((1, 3, S, S), seed=2),
                bg_img=synth.smooth_image((1, 3, S, S), seed=3))


# ----------------------------------------------------------------------------------------------------------------------
# clocks sampling during the timed region
# ----------------------------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return None
        self.proc.terminate()
        time.sleep(0.05)
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        if not sm:
            return None
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for j, n in enumerate(names) if any(len(r) > 2 + j and r[2 + j] == "Active" for r in self.rows)]
        mx = max(int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit())
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": mx, "reasons": reasons, "samples": len(sm)}


# ----------------------------------------------------------------------------------------------------------------------
# CPU baseline / reference arm: the oracle port of the reference path on the host cores
# ----------------------------------------------------------------------------------------------------------------------
def host_cores():
    """Host threads this process may really use: scheduler affinity capped by the cgroup CPU quota (a container that
    sees 128 CPUs but is throttled to a few would otherwise oversubscribe and run far slower)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if quota != "max":
            n = max(1, min(n, int(float(quota) / float(period) + 0.5)))
    except (OSError, ValueError):
        pass
    return n


def cpu_frames_per_sec(args, wl, n_frames, repeats=1, keep=None, frames=None):
    """Oracle port over `frames` (default: the first n_frames of the clip).  `keep` (a dict) receives, per frame index,
    the oracle's fim, float composite and uint8 BGR frame — what the `parity` block compares the GPU frames with."""
    import numpy as np
    import torch
    from oracle import flow_ref, generator_ref, weights
    cores = int(os.environ.get("IPER_CPU_THREADS", "0")) or host_cores()
    torch.set_num_threads(cores)
    S, tpl = args.size, wl["tpl"]
    sd = weights.synth_state_dict(0)
    src_f2pts, sfim, _ = flow_ref.render_fim_wim(wl["scams"], wl["sverts"], tpl["faces"], S)
    scond = flow_ref.encode_fim(sfim, tpl["map_fn"])
    src_inputs = torch.from_numpy(np.concatenate([wl["src_img"], scond], 1)[None])
    bg = torch.from_numpy(wl["bg_img"])
    with torch.no_grad():
        se, sr = generator_ref.forward_src(sd, src_inputs)                 # one-time per source, untimed
        times = []
        for _ in range(repeats):
            t0 = time.perf_counter()
            for i in (range(n_frames) if frames is None else frames):
                fi = flow_ref.frame_inputs(wl["cams"][i:i + 1], wl["verts"][i:i + 1], tpl["faces"], tpl["map_fn"],
                                           tpl["f_uvs2img"], wl["uv_img"], src_f2pts, S)
                img, mask = generator_ref.forward_tsf(sd, torch.from_numpy(fi["tsf_inputs"]), se, sr,
                                                      torch.from_numpy(fi["Tst"]))
                pred = generator_ref.composite(img, mask, bg)
                u8 = ((pred + 1) / 2.0 * 255).clamp(0, 255).to(torch.uint8)
                if keep is not None:
                    keep[int(i)] = dict(fim=fi["fim"][0], pred=pred[0].numpy(),
                                        u8=u8[0].numpy()[::-1].transpose(1, 2, 0))      # BGR HWC like the engine's frames
            times.append(time.perf_counter() - t0)
    return n_frames / min(times), cores, times


def run_reference(args):
    """Reference arm: the reference's OWN classes on the host cores when the staged tree (oracle/_ref) is present —
    iPERCore.models.imitator.Imitator.source_setup (untimed, once) + .inference over a bounded sample of target poses per
    step — otherwise the oracle port.  No kernel, model or engine of ipercore_b200 is on this path."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    from oracle import ref_runtime as rr
    cores = int(os.environ.get("IPER_CPU_THREADS", "0")) or host_cores()
    torch.set_num_threads(cores)
    sample = 2 if args.size >= 512 else 4
    t_start = time.perf_counter()
    if rr.available():
        import contextlib
        import tempfile
        work = tempfile.mkdtemp(prefix="iper_ref_")
        opt, model = rr.make_opt(work, image_size=args.size, num_source=args.ns)
        with contextlib.redirect_stdout(sys.stderr):      # the reference prints progress to stdout; ours is ONE json line
            im = rr.build_imitator(opt, "cpu")
        src_smpl, tgt = rr.synthetic_clip(model, sample, ns=args.ns)
        im.source_setup(rr.write_source_images(work, args.ns, args.size), src_smpl, masks=None, bg_img=None, offsets=0,
                        links_ids=None)
        times = []
        for it in range(max(args.warmup, 0) + max(args.steps, 1)):
            t0 = time.perf_counter()
            outs = im.inference(tgt, cam_strategy="smooth", output_dir="", prefix="pred_", verbose=False)
            if it >= max(args.warmup, 0):
                times.append(time.perf_counter() - t0)
        assert len(outs) == sample and outs[0].shape == (3, args.size, args.size)
        kind = "reference"
        desc = ("the reference's own iPERCore Imitator.inference (staged tree oracle/_ref: SMPLH LBS, SMPLRenderer + "
                "FlowComposition, AttentionLWBGenerator, torch fp32 on %d host threads; neural_renderer's rasteriser = host C "
                "oracle; synthetic SMPLH pkl / checkpoint), %d target poses per step, source_setup untimed" % (cores, sample))
    else:
        wl = make_workload(args, 0)
        for _ in range(max(args.warmup, 0) and 1):
            cpu_frames_per_sec(args, wl, 1)
        _, cores, times = cpu_frames_per_sec(args, wl, sample, repeats=max(args.steps, 1))
        kind = "port"
        desc = "oracle port (CPU restatement of raster+flow+AttLWB-SPADE forward_tsf, torch fp32), %d frames of the " \
               "300-pose clip per step" % sample
    fps = sample * len(times) / sum(times)
    line = {"impl": "reference", "metric": "motion_imitation_frames_per_sec", "value": fps, "unit": "frames/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * sum(times) / len(times),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config_block(args, 0),
            "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": cores, "kind": kind, "sample": desc},
            "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "wall_s": time.perf_counter() - t_start}
    print(json.dumps(line))


def gpu_library_baseline(args, dev, wl, render, src_inputs, src_f2pts):
    """The kernels to beat: the reference's own AttentionLWBGenerator.forward_tsf on torch/cuDNN on this GPU (staged tree),
    in the reference's bs=1 per-frame loop (imitator.py:341-380) and batched, TF32 (torch default), bf16 autocast and strict
    fp32.  Generator only — the reference's rasteriser extension is not available; untimed side leg, rank 0."""
    import torch
    from oracle import ref_runtime as rr
    if not rr.available():
        return {"unavailable": "reference tree not staged (oracle/_ref)"}
    net = rr.reference_generator(0, dev)
    S, ns = args.size, args.ns
    t = lambda a: torch.from_numpy(a).to(dev)
    fi = render.frame_inputs(t(wl["cams"][:16]), t(wl["verts"][:16]), t(wl["uv_img"]), src_f2pts)
    out = {"what": "reference AttentionLWBGenerator.forward_tsf (torch %s / cuDNN), %dx%d, ns=%d, generator only" %
                   (torch.__version__, S, S, ns)}
    with torch.no_grad():
        enc, res = net.forward_src(src_inputs, only_enc=True)

        def loop(bs, iters, autocast):
            e = [x.repeat(bs, 1, 1, 1) for x in enc]; r = [x.repeat(bs, 1, 1, 1) for x in res]
            ti, Ts = fi["tsf_inputs"][:bs].contiguous(), fi["Tst"][:bs].contiguous()
            def once():
                if autocast:
                    with torch.autocast("cuda", dtype=torch.bfloat16):
                        return net.forward_tsf(ti, e, r, Ts)
                return net.forward_tsf(ti, e, r, Ts)
            for _ in range(3):
                once()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize(dev); e0.record()
            for _ in range(iters):
                once()
            e1.record(); torch.cuda.synchronize(dev)
            return bs * iters / (e0.elapsed_time(e1) * 1e-3)

        for name, tf32, ac in (("tf32", True, False), ("bf16_autocast", True, True), ("fp32", False, False)):
            torch.backends.cudnn.allow_tf32 = tf32; torch.backends.cuda.matmul.allow_tf32 = tf32
            out[name] = {"bs1_loop_fps": loop(1, 20, ac), "bs16_fps": loop(16, 3, ac)}
        torch.backends.cudnn.allow_tf32 = True
    del net
    torch.cuda.empty_cache()
    return out


def run_train(args):
    """BASELINE.json configs[4]: 512x512 training step (G + D + VGG perceptual) in bf16, one sample per rank, gradients averaged with
    bucketed flat NCCL all-reduces overlapped with backward (ipercore_b200/train.py).  A side benchmark: the driver's headline
    is the default --config imitate.  value = training samples per second over all ranks."""
    import numpy as np
    import torch
    import torch.distributed as dist
    from ipercore_b200 import _lib, train
    from ipercore_b200.generator import AttentionLWBGenerator
    from oracle import weights
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    S, ns = args.size, args.ns
    net = AttentionLWBGenerator(CFG)
    net.load_state_dict(weights.synth_state_dict(0), strict=True)
    step = train.LWGTrainStep(net, dev, distributed=world > 1, graph=not args.no_graph)
    g = torch.Generator().manual_seed(100 + rank)
    r = lambda *s: (torch.rand(*s, generator=g) * 2 - 1).to(dev)
    batch = dict(bg_inputs=torch.cat([r(1, 1, 3, S, S), (r(1, 1, 1, S, S) > 0).float()], 2), src_inputs=r(1, ns, 6, S, S),
                 tsf_inputs=r(1, 1, 6, S, S), Tst=r(1, 1, ns, S, S, 2), real_src=r(1, ns, 3, S, S), real_tsf=r(1, 1, 3, S, S),
                 real_bg=r(1, 3, S, S), body_mask=(r(1, ns + 1, 1, S, S) > 0).float())

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    for _ in range(max(args.warmup, 1) + (3 if not args.no_graph else 0)):     # graph mode: 2 eager steps + the capture come first
        out = step.step(batch)
    sampler = ClockSampler(local) if rank == 0 else None
    barrier()
    n0 = _lib.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if sampler:
        sampler.start()
    e0.record()
    for _ in range(args.steps):
        out = step.step(batch)
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    if args.dump_outputs and rank == 0:     # the losses the last timed step returned, one float64 scalar per term
        os.makedirs(args.dump_outputs, exist_ok=True)
        for k, v in out.items():
            np.save(os.path.join(args.dump_outputs, "loss_%s.npy" % k), np.asarray(float(v), dtype=np.float64))
    if world > 1:
        t = torch.tensor([ms], device=dev); dist.all_reduce(t, op=dist.ReduceOp.MAX); ms = float(t)
    clocks = sampler.stop() if sampler else None
    if rank == 0:
        n_g = sum(p.numel() for p in step.G.parameters()); n_d = sum(p.numel() for p in step.D.parameters())
        line = {"metric": "lwg_training_samples_per_sec", "value": world * args.steps / (ms * 1e-3), "unit": "samples/s",
                "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
                "config": {"workload": "LWG training step %dx%d: G (AttLWB-SPADE) + D (patch_global) + VGG19 perceptual, batch 1 per GPU, "
                                       "ns=%d, nt=1 (BASELINE.json configs[4])" % (S, S, ns),
                           "kernels": "every convolution of G, D and VGG19 (stride 1 / 2 / transposed: fwd, dgrad, wgrad, bias grad) on tcgen05 bf16, "
                                      "warp, attention combine, instance norm / SPADE fwd + bwd, fused Adam + weight repack; pooling and losses are ATen",
                           "cuda_graph": not args.no_graph,
                           "allreduce": "bucketed flat NCCL all-reduce of %d G + %d D gradients, overlapped with backward" % (n_g, n_d)},
                "gpu_launches": int(args.steps * step.launches_per_step) if step._graph is not None else int(_lib.launch_count() - n0),
                "clocks": clocks,
                "losses": {k: float(v) for k, v in out.items()}}
        print(json.dumps(line), flush=True)
    if world > 1:
        # the captured graph holds NCCL work: tearing the communicator down under it hung the launcher once (2-GPU session);
        # drop the graph, drain, agree that everyone is done, and leave without running the communicator's destructor
        step._graph = None
        torch.cuda.synchronize(dev)
        dist.barrier()
        torch.cuda.synchronize(dev)
        sys.stdout.flush(); sys.stderr.flush()
        os._exit(0)


def config_block(args, launches):
    return {"workload": "run_imitator %dx%d: 1 source set (ns=%d) -> %d synthetic target SMPL poses per GPU "
                        "(BASELINE.json configs[1])" % (args.size, args.size, args.ns, args.frames),
            "image_size": args.size, "num_source": args.ns, "frames_per_step_per_gpu": args.frames, "batch": args.batch,
            "precision": args.precision, "cuda_graph": not args.no_graph, "streams": args.streams,
            "l2": "per-step working set (activations of %d-frame batches, several GB) exceeds the 126 MB L2" % args.batch,
            "weights": "synthetic (oracle/weights.py), reference 221-tensor layout"}


# ----------------------------------------------------------------------------------------------------------------------
def main():
    args = parse()
    if args.impl == "reference":
        return run_reference(args)
    if args.config == "train":
        return run_train(args)
    import numpy as np
    import torch
    import torch.distributed as dist
    from ipercore_b200 import _lib, ops
    from ipercore_b200.engine import FrameEngine
    from ipercore_b200.generator import AttentionLWBGenerator
    from ipercore_b200.renders import SMPLRenderer
    from oracle import weights

    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    wl = make_workload(args, rank)
    tpl, S, ns = wl["tpl"], args.size, args.ns
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)

    render = SMPLRenderer(image_size=S, tables=tpl, has_front=True, top_k=3).to(dev)
    gen = AttentionLWBGenerator(CFG, precision=args.precision)
    gen.load_state_dict(weights.synth_state_dict(0), strict=True)
    gen = gen.to(dev).eval()
    # one-time per source: geometry of the source views -> f2pts + cond; input_G_src = cat[src_img, cond]
    src_f2pts, sfim, _ = render.render_fim_wim(t(wl["scams"]), t(wl["sverts"]))
    scond, _ = render.encode_fim(fim=sfim)
    src_inputs = torch.cat([t(wl["src_img"]), scond], 1)[None]
    engines = []
    for _ in range(max(args.streams, 1)):
        e = FrameEngine(gen, render, batch=args.batch, use_graph=not args.no_graph, device=dev)
        e.set_source(src_inputs, t(wl["uv_img"]), t(wl["bg_img"]), src_f2pts)
        engines.append(e)
    eng = engines[0]

    T, B = args.frames, args.batch
    cams_d, verts_d = t(wl["cams"]), t(wl["verts"])
    cams_h = torch.from_numpy(wl["cams"]).pin_memory(); verts_h = torch.from_numpy(wl["verts"]).pin_memory()
    out_h = torch.empty((T, S, S, 3), dtype=torch.uint8).pin_memory()
    out_d = torch.empty((T, S, S, 3), dtype=torch.uint8, device=dev)
    nb = (T + B - 1) // B
    cur = torch.cuda.current_stream(dev)

    def step_device():
        for i in range(nb):
            lo, hi = i * B, min((i + 1) * B, T)
            e = engines[i % len(engines)]
            u8 = e.run_batch_device(cams_d[lo:hi], verts_d[lo:hi])
            with torch.cuda.stream(e.compute):
                out_d[lo:hi].copy_(u8[:hi - lo], non_blocking=True)
        for e in engines:
            cur.wait_stream(e.compute)

    def step_e2e():
        eng.synthesize(cams_h, verts_h, out=out_h)

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def timed(fn, steps, sampler=None):
        barrier()
        for e in engines:
            e.compute.wait_stream(cur); e.copy.wait_stream(cur)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        if sampler:
            sampler.start()
        w0 = time.perf_counter()
        e0.record(cur)
        for e in engines:
            e.compute.wait_event(e0); e.copy.wait_event(e0)
        for _ in range(steps):
            fn()
        e1.record(cur)
        barrier()
        wall = time.perf_counter() - w0
        ms = e0.elapsed_time(e1)
        if world > 1:
            tt = torch.tensor([ms], device=dev)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            ms = float(tt)
        return ms, wall

    if args.profile_batch:
        eng.use_graph = False
        eng.run_batch_device(cams_d[:B], verts_d[:B])          # warm-up (packs weights, fills caches)
        torch.cuda.synchronize(dev)
        torch.cuda.profiler.start()
        eng.run_batch_device(cams_d[:B], verts_d[:B])
        torch.cuda.synchronize(dev)
        torch.cuda.profiler.stop()
        print(json.dumps({"profile_batch": B, "launches_per_batch": eng.launches_per_batch}))
        return
    for _ in range(max(args.warmup, 1)):
        step_device()
    sampler = ClockSampler(local) if rank == 0 else None
    launches0 = _lib.launch_count()
    ms, wall = timed(step_device, args.steps, sampler)
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:     # out_d holds every frame of the last timed step (rank 0's clip)
        dump_frames(args.dump_outputs, out_d)
    fps = world * T * args.steps / (ms * 1e-3)
    for _ in range(1):
        step_e2e()
    ms_e2e, _ = timed(step_e2e, args.steps)
    fps_e2e = world * T * args.steps / (ms_e2e * 1e-3)
    launches = eng.launches_per_batch * nb * args.steps if eng.graph else _lib.launch_count() - launches0

    # ---- parity of the frames the timed e2e region just produced (rank 0): oracle port on a sample of frames ----------
    # out_h holds every uint8 frame of the last e2e step; eng.last_pred the float composites of its last batch.
    cpu, parity = None, None
    if rank == 0 and not args.no_parity:
        try:
            keep = {}
            if world == 1 and not args.no_cpu_baseline:     # the cpu_baseline leg already runs the oracle: keep its frames
                v, cores, _ = cpu_frames_per_sec(args, wl, args.cpu_frames, keep=keep)
                cpu = {"value": v, "unit": "frames/s", "cores": cores, "kind": "port",
                       "sample": "first %d frames of the 300-pose clip through the oracle port (CPU restatement of raster + "
                                 "flow + forward_tsf + composite, torch fp32, all host threads); source setup untimed" % args.cpu_frames}
            last_lo = (nb - 1) * B
            extra = sorted({last_lo, T - 1, min(B - 1, T - 1), min(B, T - 1)} - set(keep))   # batch edges + the last batch
            cpu_frames_per_sec(args, wl, 0, keep=keep, frames=extra)
            idx = sorted(keep)
            got_u8 = out_h.numpy()
            code = max(int(np.abs(got_u8[i].astype(np.int32) - keep[i]["u8"].astype(np.int32)).max()) for i in idx)
            frac = float(np.mean([(got_u8[i] != keep[i]["u8"]).mean() for i in idx]))
            sel = torch.tensor(idx, device=dev)
            fi = render.frame_inputs(cams_d[sel].contiguous(), verts_d[sel].contiguous(), eng.src["uv_img"], eng.src["src_f2pts"],
                                     want_fim=True)
            fim_equal = all(np.array_equal(fi["fim"][k].cpu().numpy(), keep[i]["fim"]) for k, i in enumerate(idx))
            lastp = eng.last_pred.float().cpu().numpy()      # composites of the last batch of the last e2e step
            fl = [i for i in idx if i >= last_lo]
            max_abs = max(float(np.abs(lastp[i - last_lo] - keep[i]["pred"]).max()) for i in fl)
            parity = {"frames": len(idx), "frame_ids": idx, "max_abs": max_abs, "max_abs_frames": fl, "tolerance": 1e-3,
                      "u8_max_code_diff": code, "u8_frac_differing": frac, "fim_equal": bool(fim_equal),
                      "ok": bool(fim_equal and max_abs <= 1e-3 and code <= 1),
                      "against": "oracle port (CPU restatement pinned to the reference's own modules by tests/golden) on the "
                                 "uint8 frames of the last timed e2e step (all sampled frames) and the float composites of its "
                                 "last batch; face-index maps re-rendered for the sampled frames"}
            if not parity["ok"]:
                sys.stderr.write("bench.py: PARITY FAILED %s\n" % json.dumps(parity))
        except Exception as exc:     # a checker failure must be visible in the line, never lose the measurement
            parity = {"ok": False, "error": "%s: %s" % (type(exc).__name__, exc)}

    # ---- output stage: the same e2e pass with PNG files written like Imitator.inference does (pred_%08d.png), encodes
    #      overlapped with the next batch (engine.synthesize_stream + patch.FrameWriter); rank 0, one pass ----------------
    e2e_png = None
    if rank == 0 and world == 1 and not args.no_png:
        import shutil
        import tempfile
        from ipercore_b200.patch import FrameWriter
        out_dir = tempfile.mkdtemp(prefix="iper_png_", dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
        try:
            def feed(lo, hi):
                return cams_h[lo:hi].to(dev, non_blocking=True), verts_h[lo:hi].to(dev, non_blocking=True)
            for rep in range(2):                  # first pass warms the pool / page cache
                writer = FrameWriter(T, out_dir, "pred_", workers=host_cores())
                torch.cuda.synchronize(dev)
                w0 = time.perf_counter()
                eng.synthesize_stream(T, feed, writer.sink)
                paths = writer.close()
                torch.cuda.synchronize(dev)
                w_png = time.perf_counter() - w0
            nbytes = sum(os.path.getsize(p_) for p_ in paths)
            e2e_png = {"value": T / w_png, "unit": "frames/s", "frames": T, "workers": host_cores(),
                       "png_bytes_per_frame": nbytes // T, "timing": "host wall clock around one whole clip incl. the last file",
                       "files": "pred_%08d.png (cv2.imwrite, uint8 BGR), " + ("tmpfs" if out_dir.startswith("/dev/shm") else "tmp dir")}
        except Exception as exc:
            e2e_png = {"error": "%s: %s" % (type(exc).__name__, exc)}
        finally:
            shutil.rmtree(out_dir, ignore_errors=True)

    # ---- strong scaling: ONE clip of T frames split over the ranks (engine.shard_range), batch sized to the shard -------
    strong = None
    if world > 1 and not args.no_strong:
        from ipercore_b200.engine import balanced_batch, shard_range
        wl0 = wl if rank == 0 else make_workload(args, 0)       # every rank takes a contiguous shard of rank 0's clip
        lo_s, hi_s = shard_range(T, rank, world)
        Bs = balanced_batch(hi_s - lo_s, B)
        es = FrameEngine(gen, render, batch=Bs, use_graph=not args.no_graph, device=dev)
        es.src = eng.src
        cams_s, verts_s = t(wl0["cams"][lo_s:hi_s]), t(wl0["verts"][lo_s:hi_s])
        n_s = hi_s - lo_s

        def step_strong():
            for b0 in range(0, n_s, Bs):
                b1 = min(b0 + Bs, n_s)
                u8 = es.run_batch_device(cams_s[b0:b1], verts_s[b0:b1])
                with torch.cuda.stream(es.compute):
                    out_d[b0:b1].copy_(u8[:b1 - b0], non_blocking=True)
            cur.wait_stream(es.compute)

        engines.append(es)
        for _ in range(max(args.warmup, 1)):
            step_strong()
        ms_s, _ = timed(step_strong, args.steps)
        engines.pop()
        strong = {"value": T * args.steps / (ms_s * 1e-3), "unit": "frames/s", "frames_total": T, "frames_rank0": n_s,
                  "batch": Bs, "ms_per_step": ms_s / args.steps,
                  "note": "one %d-frame clip split contiguously over %d ranks, no collective; max over ranks" % (T, world)}

    lib_base = None
    if rank == 0 and world == 1 and not args.no_lib_baseline:
        try:
            lib_base = gpu_library_baseline(args, dev, wl, render, src_inputs, src_f2pts)
        except Exception as exc:   # a side leg must never take the bench line down
            lib_base = {"unavailable": "%s: %s" % (type(exc).__name__, exc)}

    # ---- roofline of the conv stack: CUDA events around every conv_gemm launch of one (un-graphed) batch ----
    roof = None
    if rank == 0:
        recs = []
        orig = ops.conv_gemm

        def timed_conv(a, wpack, mode, ksize, rows, block_n, epi, **kw):  # noqa: E306
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); orig(a, wpack, mode, ksize, rows, block_n, epi, **kw); e1.record()
            phases = 4 if mode == ops.IPER_CONVT_4S2 else 1
            opix = a.N * (a.H // 2) * (a.W // 2) if mode == ops.IPER_CONV_S2 else a.N * a.H * a.W
            macs = opix * phases * rows * wpack.K
            recs.append((e0, e1, macs * {1: 1, 2: 3, 3: 2}[wpack.fmt],    # fp16-equivalent MMA work per mode
                         dict(mode=mode, ksize=ksize, rows=rows, K=wpack.K, N=a.N, H=a.H, W=a.W, epi=epi,
                              cta_pair=kw.get("cta_pair", 0))))

        other = []          # (name, e0, e1) of the non-conv launches of the same batch
        OTHER_OPS = ("raster_frames", "conv_stem", "conv_stem_tc", "stem_im2col", "warp_attention", "flow_resize", "instnorm_finalize", "pred_to_u8")
        saved = {k: getattr(ops, k) for k in OTHER_OPS if hasattr(ops, k)}

        def wrap(name, fn):  # noqa: E306
            def timed_other(*a_, **kw_):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(); out = fn(*a_, **kw_); e1.record()
                other.append((name, e0, e1))
                return out
            return timed_other

        with torch.cuda.stream(eng.compute):
            eng._step()
            ops.conv_gemm = timed_conv
            for k, fn in saved.items():
                setattr(ops, k, wrap(k, fn))
            try:
                s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s0.record(); eng._step(); s1.record()
            finally:
                ops.conv_gemm = orig
                for k, fn in saved.items():
                    setattr(ops, k, fn)
            torch.cuda.synchronize(dev)
        conv_ms = sum(r[0].elapsed_time(r[1]) for r in recs)
        step_ms = s0.elapsed_time(s1)
        exec_flops = 2.0 * sum(r[2] for r in recs)
        if args.dump_layers:     # per-launch table of the conv stack (ms, executed fp16-equivalent TFLOP/s)
            rows_ = [dict(r[3], ms=r[0].elapsed_time(r[1]), exec_tflops=2.0 * r[2] / (r[0].elapsed_time(r[1]) * 1e-3) / 1e12)
                     for r in recs]
            agg = {}
            for name, e0, e1 in other:
                agg.setdefault(name, [0, 0.0]); agg[name][0] += 1; agg[name][1] += e0.elapsed_time(e1)
            with open(args.dump_layers, "w") as f:
                json.dump(rows_, f, indent=0)
            with open(args.dump_layers + ".other.json", "w") as f:
                json.dump({k: dict(launches=v[0], ms=v[1]) for k, v in agg.items()}, f, indent=1)
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except OSError:
            pass
        peak = peaks.get("bf16_tflops_sustained", 1400.0)
        alg = FLOPS_PER_FRAME_512 * (S / 512.0) ** 2 * (1 + (ns - 2) * 9.66 / 285.93) * B
        ach = alg / (conv_ms * 1e-3) / 1e12
        traffic = None
        try:
            # DRAM bytes of the conv launches of one batch (ncu --set full capture, per frame x frames per batch); like
            # `achieved` it covers the whole conv stack of a batch, the unit the roofline is stated for
            per_frame = json.load(open(os.path.join(ROOT, "profiles", "conv_traffic.json"))).get("dram_bytes_per_frame")
            traffic = per_frame * B * (S / 512.0) ** 2 if per_frame else None
        except (OSError, ValueError):
            pass
        roof = {"bound": "tensor", "kernel": "conv_halo_pair_kernel / conv_gemm_pair_kernel (tcgen05 cta_group::2 implicit GEMM, %d launches per %d-frame batch)" % (len(recs), B),
                "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak,
                "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained (measured)" if peaks else "fallback 1.4 PFLOP/s sustained",
                "algorithmic_flops_per_batch": alg, "executed_tflops": exec_flops / (conv_ms * 1e-3) / 1e12,
                "executed_flops_note": "fp16-equivalent MMA work: fp16x2 = 3 MMAs per K step, fp16f8 = 1 fp16 + 2 e4m3 (2x rate) = 2; fk/fv hoisted to once-per-source",
                "conv_ms_per_batch": conv_ms, "batch_ms_ungraphed": step_ms, "conv_share_of_step": conv_ms / step_ms,
                "traffic": traffic,
                "traffic_note": "dram__bytes_read+write of the batch's conv launches (profiles/conv_traffic.json, ncu --set full); "
                                "the stack is tensor-bound, DRAM runs at ~1.4 TB/s"}

    if cpu is None and rank == 0 and world == 1 and not args.no_cpu_baseline:
        v, cores, _ = cpu_frames_per_sec(args, wl, args.cpu_frames)
        cpu = {"value": v, "unit": "frames/s", "cores": cores, "kind": "port",
               "sample": "first %d frames of the 300-pose clip through the oracle port (CPU restatement of raster + "
                         "flow + forward_tsf + composite, torch fp32, all host threads); source setup untimed" % args.cpu_frames}

    if rank == 0:
        line = {"metric": "motion_imitation_frames_per_sec", "value": fps, "unit": "frames/s", "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None,
                "dtype": {"fp16x2": "f16x2 (split fp16 operands, fp32 accumulate)", "fp16": "f16 (fp32 accumulate)",
                          "fp16f8": "f16 + e4m3 cross terms (fp32 accumulate)",
                          "mixed": "f16x2, SPADE convs single-pass f16 (opt-in, outside the parity tolerance)"}[args.precision],
                "data": "synthetic", "config": config_block(args, launches),
                "e2e": {"value": fps_e2e, "unit": "frames/s", "h2d_bytes_per_step": int(cams_h.numel() * 4 + verts_h.numel() * 4),
                        "d2h_bytes_per_step": int(out_h.numel()), "ms_per_step": ms_e2e / args.steps},
                "gpu_launches": int(launches), "clocks": clocks, "roofline": roof, "cpu_baseline": cpu,
                "parity": parity, "strong": strong, "e2e_png": e2e_png,
                "gpu_library_baseline": lib_base,
                "wall_s_timed_region": wall}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
