#!/usr/bin/env python
"""Benchmark of the per-frame inference hot path (BASELINE.json metric: frames/s @256x256, bs16).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--batch 16] [--size 256] [--dump-outputs DIR]

One *step* = one pass of the hot path over one batch of B synthetic target frames per GPU:
fused correspondence (raster + cond + T + image warp) -> ImpersonatorGenerator.inference on the
tcgen05 conv engine (fp16f8 / fp16x3 parity modes) -> composite.  N > 1: one process per GPU (torchrun),
frames sharded across ranks (weak scaling), ONE NCCL broadcast of weights + source state at init,
no per-step collective.  Prints ONE JSON line on rank 0.

``value``   whole-job frames/s with inputs already resident in HBM (CUDA events, max over ranks).
``e2e``     the same metric through the reference-facing API (Imitator.inference_by_smpls) with HOST
            inputs (pinned SMPL vectors) and HOST outputs (float32 HxWx3 frames), copies inside the timer.
``roofline`` conv-engine kernels (tensor bound): algorithmic FLOPs / CUDA-event time of those launches.
``cpu_baseline`` the oracle port (C rasterizer restatement + torch-CPU generator restatement, i.e. the
            same ATen CPU ops the reference modules call) on the host cores, bounded sample, rank 0, N=1.
``--impl reference`` times that CPU path as the reference arm (the reference tree itself does not exist
            on the GPU box; its CUDA rasterizer has no CPU path at all).
``--dump-outputs DIR`` writes what the last timed step returned -- the generated frames, float32 [B,3,H,W] -- as
            DIR/pred.npy (rank 0's frames; the first frames only beyond DUMP_BYTES).  The inputs are seeded, so two builds
            run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FLOPS_PER_FRAME_TC = None   # filled from the conv plans (algorithmic 2*MAC of the tensor-core layers)
REF_INFERENCE_GFLOP = 105.579   # BASELINE.md section 2: generator.inference per frame @256^2
DUMP_BYTES = 64 << 20           # --dump-outputs writes at most this much


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=16)
    ap.add_argument("--size", type=int, default=256)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip roofline instrumentation / fast-mode legs")
    ap.add_argument("--profile-range", action="store_true", help="cudaProfilerStart/Stop around the timed steps (ncu --profile-from-start off)")
    ap.add_argument("--steady-steps", type=int, default=400, help="length of the extra steady-state leg (N=1; 0 = skip)")
    ap.add_argument("--no-parity", action="store_true", help="skip the oracle check of one step (outside the timed region)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the frames the last timed step returned as DIR/pred.npy")
    return ap.parse_args()


# --------------------------------------------------------------------------------------------
# clocks: nvidia-smi sampled DURING the timed region
# --------------------------------------------------------------------------------------------
class ClockSampler(object):
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)
        self.proc.terminate()
        sm, mx, reasons, pw = [], [], set(), []
        for ln in self.lines:
            p = [t.strip() for t in ln.split(",")]
            if len(p) < 7:
                continue
            try:
                sm.append(float(p[0])); mx.append(float(p[1])); pw.append(float(p[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


# --------------------------------------------------------------------------------------------
# CPU reference arm / cpu_baseline: oracle port on the host cores
# --------------------------------------------------------------------------------------------
def cpu_reference_setup(size):
    import torch
    from impersonator_b200 import synthetic as S
    from impersonator_b200.generator import ImpersonatorGenerator
    from oracle import generator_ref as G, nmr_ref, raster, smpl_ref
    torch.set_grad_enabled(False)
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    v, f = S.uv_sphere()
    tabs = S.synthetic_tables()
    src_img = S.synthetic_source(size)
    tmpl = ImpersonatorGenerator(bg_dim=4, src_dim=6, tsf_dim=6, repeat_num=6).state_dict()
    sd = S.fill_state_dict(tmpl, seed=0)
    body = smpl_ref.model_tensors(S.synthetic_smpl_model(seed=3))
    det = smpl_ref.get_details(body, S.synthetic_smpl_params(1, seed=5))
    cam, verts = det["cam"], det["verts"]
    f2v, fim, _ = nmr_ref.render_fim_wim(cam, verts, f, size)
    p2v = nmr_ref.src_p2verts(f2v)
    src_inputs = torch.cat([src_img, nmr_ref.encode_fim(fim, tabs["map_fn"])], dim=1)
    feats = G.encode_src(src_inputs, sd)
    bg = torch.zeros(1, 3, size, size)
    state = dict(v=v, f=f, tabs=tabs, src_img=src_img, sd=sd, p2v=p2v, feats=feats, bg=bg, size=size,
                 cores=max(cores, raster.num_threads()))

    frame_sets = {}

    def run(nframes, seed):
        if (nframes, seed) not in frame_sets:                       # synthetic input generation is not timed work
            frame_sets[(nframes, seed)] = S.synthetic_smpl_params(nframes, seed=seed)
        det = smpl_ref.get_details(body, frame_sets[(nframes, seed)])     # SMPL vectors in, like the e2e leg
        cam, verts = det["cam"], det["verts"]
        c = nmr_ref.correspond(cam, verts, f, tabs["map_fn"], p2v, src_img, size)
        pred, _, _ = G.imitator_forward(bg, feats, c["tsf_inputs"], c["T"], sd)
        return pred
    state["run"] = run
    # "all the host threads it can use": more threads than the work can feed only slows oneDNN / the
    # pthread rasterizer down, so pick the fastest of a few thread counts on one frame each.
    best = None
    run(1, 90)
    for nt in sorted({cores, min(cores, 64), min(cores, 32), min(cores, 16), min(cores, 8)}, reverse=True):
        torch.set_num_threads(nt)
        raster._cpu_lib().lwb_oracle_set_num_threads(nt)
        run(1, 90)
        dts = []
        for _ in range(3):                                          # median of 3: one sample per candidate was noisy
            t0 = time.time()
            run(1, 90)
            dts.append(time.time() - t0)
        dt = sorted(dts)[1]
        if best is None or dt < best[0]:
            best = (dt, nt)
    torch.set_num_threads(best[1])
    raster._cpu_lib().lwb_oracle_set_num_threads(best[1])
    state["cores"] = best[1]
    state["cores_available"] = cores
    state["sec_per_frame"] = best[0]
    return state


def cpu_baseline(size, frames_per_rep=4, reps=3):
    st = cpu_reference_setup(size)
    st["run"](frames_per_rep, 200)                              # warm-up + input generation (untimed)
    t0 = time.time()
    for r in range(reps):
        st["run"](frames_per_rep, 200)
    dt = time.time() - t0
    return {"value": frames_per_rep * reps / dt, "unit": "frames/s", "cores": st["cores"], "cores_available": st["cores_available"], "kind": "port",
            "sample": "%d frames (%d x batch %d) of the same workload: C rasterizer restatement (pthreads) + torch-CPU "
                      "(oneDNN fp32) restatement of nmr glue + generator.inference + composite, %.1f s"
                      % (frames_per_rep * reps, reps, frames_per_rep, dt)}


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    st = cpu_reference_setup(args.size)
    # one full batch per step when the whole run fits ~4 minutes, else a bounded sample of the batch
    budget = 240.0 / max(1, args.steps + max(args.warmup, 1))
    per_step = int(max(2, min(args.batch, budget / max(st["sec_per_frame"], 1e-3))))
    for i in range(max(args.warmup, 1)):
        st["run"](per_step, 300 + (i % 2))
    t0 = time.time()
    for i in range(args.steps):
        st["run"](per_step, 300 + (i % 2))
    dt = time.time() - t0
    fps = per_step * args.steps / dt
    line = {"impl": "reference", "metric": "frames/sec @256x256 (per-frame inference hot path)", "value": fps, "unit": "frames/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args, per_step),
            "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": st["cores"], "kind": "port",
                             "cores_available": st["cores_available"],
                             "sample": "%d frames per step (%s of the batch-%d workload), ONE process, CPU oracle port: "
                                       "C rasterizer restatement + torch-CPU generator restatement"
                                       % (per_step, "the full batch" if per_step == args.batch else "bounded sample", args.batch)},
            "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


def workload_config(args, frames_per_step=None):
    return {"workload": "BASELINE configs[2]: batch-%d motion-imitation inference loop (SMPL raster + correspondence + LWB + "
                        "generator.inference + composite; e2e adds SMPL LBS from 85-float vectors), %dx%d, synthetic SMPL-shaped body V=6890 F=13776, random-init "
                        "ImpersonatorGenerator (97.45 M params)" % (args.batch, args.size, args.size),
            "frames_per_step_per_gpu": frames_per_step if frames_per_step is not None else args.batch,
            "image_size": args.size, "precision": "LWB_PRECISION=%s: fp16 hi/lo operand split on tcgen05, fp32 accumulate (parity-gated 1e-3 vs fp32)"
                         % os.environ.get("LWB_PRECISION", "fp16f8 (default)"),
            "parallelism": "frames sharded, dp%d, no per-step collective" % args.gpus,
            "engine": {k: os.environ.get(k, d) for k, d in (("LWB_STREAMS", "2 (default)"), ("LWB_GRAPH", "1 (default)"),
                                                              ("LWB_YHALO", "1 (default)"), ("LWB_TC_HEADS", "1 (default)"),
                                                              ("LWB_CONVT_MERGE", "1 (default)"), ("LWB_FUSE_NORM", "0 (default)"),
                                                              ("LWB_ALIGN_CORNERS", "1 (default, torch-1.2 grid_sample)"))},
            "l2": "per-step working set (~2 GB of activations at batch 16) >> 126 MB L2; inputs rotate over 4 frame sets"}


def parity_check(imitator, step_device, dev_set, faces, tabs, src_img, src_theta, size, B, frames=(0, -1)):
    """One step of the timed workload against the CPU oracle (oracle/: checker only, never timed): the first and last
    frame of frame set 0.  The oracle consumes the vertices the LBS kernels produced (their own parity is a test), so
    that 1e-7 vertex differences cannot flip silhouette pixels of the bit-exact rasterizer."""
    import torch
    from oracle import generator_ref as G, nmr_ref
    t0 = time.time()
    sd = {k: v.detach().cpu() for k, v in imitator.generator.state_dict().items()}
    pred = step_device(0).cpu()
    cam, verts = dev_set[0].cpu(), dev_set[1].cpu()
    s_cam, s_verts = imitator.src_info["cam"].cpu(), imitator.src_info["verts"].cpu()
    f2v, sfim, _ = nmr_ref.render_fim_wim(s_cam, s_verts, faces, size)
    cond = nmr_ref.encode_fim(sfim, tabs["map_fn"])
    p2v = nmr_ref.src_p2verts(f2v)
    from impersonator_b200.imitator import morph
    bg_mask = morph(cond[:, -1:], 13, 'erode')
    bg = G.resnet_generator(torch.cat([src_img * bg_mask, bg_mask], dim=1), sd, 'bg_model')
    ft_mask = 1 - morph(cond[:, -1:], 3, 'erode')
    feats = G.encode_src(torch.cat([src_img * ft_mask, cond], dim=1), sd)
    sel = sorted({i % B for i in frames})
    c = nmr_ref.correspond(cam[sel], verts[sel], faces, tabs["map_fn"], p2v, src_img, size)
    ref, _, _ = G.imitator_forward(bg, feats, c["tsf_inputs"], c["T"], sd)
    d = (pred[sel] - ref).abs().amax(dim=(1, 2, 3)).tolist()
    return {"max_abs": max(d), "per_frame": d, "frames_checked": sel, "tol": 1e-3, "ok": bool(max(d) < 1e-3),
            "against": "CPU oracle (oracle/nmr_ref.py + raster_ref.c + generator_ref.py), outside the timed region",
            "seconds": time.time() - t0}


# --------------------------------------------------------------------------------------------
# our arm
# --------------------------------------------------------------------------------------------
def main():
    args = parse()
    if args.impl == "reference":
        return run_reference_arm(args)

    import torch
    import torch.distributed as dist
    from impersonator_b200 import _lib, kernels as K, synthetic as S
    from impersonator_b200 import generator as GEN
    from impersonator_b200.generator import ImpersonatorGenerator
    from impersonator_b200.imitator import Imitator
    from impersonator_b200.hmr import HumanModelRecovery
    from impersonator_b200.nmr import SMPLRenderer

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    _lib.require_gpu()
    torch.set_grad_enabled(False)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    B, size = args.batch, args.size
    mode = GEN.precision_mode()

    # ---- init: rank 0 owns weights + source state, ONE broadcast of a packed buffer -----------
    v, f = S.uv_sphere()
    tabs = S.synthetic_tables()
    net = ImpersonatorGenerator(bg_dim=4, src_dim=6, tsf_dim=6, repeat_num=6)
    src_img = S.synthetic_source(size)
    if rank == 0:
        net.load_state_dict(S.fill_state_dict(net.state_dict(), seed=0))
    else:
        src_img = torch.zeros_like(src_img)
    from impersonator_b200 import sharding
    bc_stats = {}
    src_img = sharding.broadcast_module(net, extras=[src_img], src=0, device=dev, stats=bc_stats)[0]      # the ONE collective
    net = net.to(dev).eval()
    render = SMPLRenderer(image_size=size, faces=f.numpy(), map_fn=tabs["map_fn"], has_front=False).to(dev)

    class Opt(object):
        image_size, batch_size, bg_model, repeat_num, cond_nc = size, B, "ORIGINAL", 6, 3
        bg_ks, ft_ks, front_warp, only_vis = 13, 3, False, False
    body = HumanModelRecovery(smpl_model=S.synthetic_smpl_model(seed=3)).to(dev)       # SMPL LBS kernels (csrc/smpl.cu)
    imitator = Imitator(Opt(), generator=net, hmr=body, render=render, device=dev)
    src_theta = S.synthetic_smpl_params(1, seed=5)[0]
    imitator.personalize("", src_smpl=src_theta.numpy(), src_img=src_img)           # once per source (untimed)
    pers = []
    for _ in range(6):
        torch.cuda.synchronize()
        t0 = time.time()
        imitator.personalize("", src_smpl=src_theta.numpy(), src_img=src_img)
        torch.cuda.synchronize()
        pers.append((time.time() - t0) * 1e3)
    personalize_ms = sorted(pers[1:])[2]                                            # median of 5 after one more warm call
    inpaint_ms = None
    if rank == 0 and not args.no_extras:
        # the DeepFill-v2 background network (opt.bg_model != 'ORIGINAL', models/imitator.py:48-52,125) on the conv engine
        from impersonator_b200.inpaintor import InpaintSANet
        inp_net = InpaintSANet(c_dim=4)
        inp_net.load_state_dict(S.fill_state_dict(inp_net.state_dict(), seed=3, conv_std=0.05))
        inp_net = inp_net.to(dev).eval()
        msk = torch.zeros(1, 1, size, size, device=dev)
        msk[:, :, size // 4:3 * size // 4, size // 3:2 * size // 3] = 1
        for _ in range(3):
            inp_net(src_img.to(dev), msk, only_x=True)
        torch.cuda.synchronize()
        i0, i1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        i0.record()
        for _ in range(10):
            inp_net(src_img.to(dev), msk, only_x=True)
        i1.record()
        torch.cuda.synchronize()
        inpaint_ms = i0.elapsed_time(i1) / 10
        del inp_net

    # per-step target frames: 4 rotating sets per rank, resident in HBM for `value`
    def thetas(seed):
        return S.synthetic_smpl_params(B, seed=seed)
    host_sets = [thetas(1000 + 17 * rank + i) for i in range(4)]
    imitator.first_cam = host_sets[0][0:1, 0:3].to(dev)
    dev_sets = []
    for th in host_sets:
        det = body.get_details(imitator.swap_smpl(imitator.src_info["cam"], imitator.src_info["shape"], th.to(dev), "smooth"))
        dev_sets.append((det["cam"].contiguous(), det["verts"].contiguous()))
    enc, res = imitator.src_info["feats"]
    bg = imitator.src_info["bg"]
    p2v, simg = imitator.src_info["p2verts"], imitator.src_info["img"]

    def step_body(cam, verts):
        out = render.correspond(cam, verts, p2v, simg)
        return net.inference(enc, res, out["tsf_inputs"], out["T"], bg=bg)[2]

    def step_eager(i):
        cam, verts = dev_sets[i % len(dev_sets)]
        return step_body(cam, verts)

    # Operand-precision policy, as Imitator.inference applies it: if the default fp16f8 mode raises a range bit on this
    # rank's frames (bit 0: |x| >= 1024, bit 2: head pre-activations beyond +-8), the rank runs fp16x3 -- `value` is
    # measured under the product's own policy on every rank, never in a mode the API would have left.
    policy_bits = 0
    for i in range(len(dev_sets)):
        step_eager(i)
        policy_bits |= net.tsf_model.range_status()
    if policy_bits & 2:
        raise SystemExit("bench: activations beyond the fp16 range on rank %d" % rank)
    if (policy_bits & 5) and mode == "fp16f8" and os.environ.get("LWB_AUTO_PRECISION", "1") != "0":
        net.set_precision("fp16x3")
        imitator.personalize("", src_smpl=src_theta.numpy(), src_img=src_img)
        enc, res = imitator.src_info["feats"]
        bg = imitator.src_info["bg"]
        p2v, simg = imitator.src_info["p2verts"], imitator.src_info["img"]
        mode = "fp16x3"
    modes_by_rank = [mode]
    if world > 1:
        modes_by_rank = [None] * world
        dist.all_gather_object(modes_by_rank, mode)

    # LWB_GRAPH (default on): the step's launch sequence is captured once and replayed (one cudaGraphLaunch per step); the
    # frame set of the step is copied device-to-device into the graph's static input (1.3 MB), still "resident in HBM"
    from impersonator_b200.graph import CapturedStep, graphs_enabled
    captured = CapturedStep(step_body, dict(cam=dev_sets[0][0], verts=dev_sets[0][1])) if graphs_enabled() else None

    def step_device(i):
        if captured is None or not captured.captured:
            return step_eager(i)
        cam, verts = dev_sets[i % len(dev_sets)]
        return captured(cam=cam, verts=verts)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    last_out = [None]

    def timed(fn, steps, warmup, collective=True, profile=False):
        """collective=False: rank-local timing (the rank-0-only extras must not enter a barrier).  profile: bracket the
        timed steps with cudaProfilerStart/Stop (--profile-range, for `ncu --profile-from-start off`).  The last step's
        output is left in last_out[0]."""
        for i in range(warmup):
            fn(i)
        if collective:
            barrier()
        else:
            torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        K.reset_launch_count()
        if profile:
            torch.cuda.profiler.start()
        e0.record()
        for i in range(steps):
            last_out[0] = fn(warmup + i)
        e1.record()
        torch.cuda.synchronize()
        if profile:
            torch.cuda.profiler.stop()
        ms = e0.elapsed_time(e1)
        launches = K.launch_count()
        if world > 1 and collective:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = t.item()
            dist.barrier()
        return ms, launches

    # ---- parity of one step against the CPU oracle, OUTSIDE every timed region (rank 0) ---------
    parity = None
    if rank == 0 and not args.no_parity:
        parity = parity_check(imitator, step_device, dev_sets[0], f, tabs, src_img.cpu(), src_theta, size, B)
        if not parity["ok"]:
            raise SystemExit("bench: parity check failed: %s" % json.dumps(parity))

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ms, launches = timed(step_device, args.steps, max(args.warmup, 3), profile=args.profile_range)
    clocks = sampler.stop() if rank == 0 else None
    fps = world * B * args.steps / (ms * 1e-3)
    if rank == 0 and args.dump_outputs:
        # copied now: a captured step returns a static buffer that the legs below overwrite
        import numpy as np
        pred = last_out[0].float().cpu().numpy()
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "pred.npy"), pred[:DUMP_BYTES // pred[0].nbytes])
    # ---- BASELINE configs[3] as written: a 64-frame stream sharded over the ranks (8 per GPU at N = 8), strong scaling:
    # total work fixed, every rank runs its 64 / N frames in chunks of at most B; time = max over ranks
    c3_frames = 64
    c3 = None
    if c3_frames % world == 0 and not args.profile_range:
        per_rank = c3_frames // world
        a0, _ = sharding.shard_range(c3_frames, rank, world)
        c3_sets = []
        for k in range(0, per_rank, B):
            nb = min(B, per_rank - k)
            th = S.synthetic_smpl_params(c3_frames, seed=4242)[a0 + k:a0 + k + nb]
            det = body.get_details(imitator.swap_smpl(imitator.src_info["cam"], imitator.src_info["shape"], th.to(dev), "smooth"))
            c3_sets.append((det["cam"].contiguous(), det["verts"].contiguous()))

        def step_c3(i):
            out = None
            for cam, verts in c3_sets:
                o = render.correspond(cam, verts, p2v, simg)
                out = net.inference(enc, res, o["tsf_inputs"], o["T"], bg=bg)[2]
            return out
        reps = 5
        ms_c3, _ = timed(step_c3, reps, 3)
        c3 = {"workload": "BASELINE configs[3]: 64-frame stream, %d frames per GPU on %d GPU(s), weights broadcast once" % (per_rank, world),
              "frames": c3_frames, "frames_per_gpu": per_rank, "ms_per_64_frames": ms_c3 / reps,
              "value": c3_frames / (ms_c3 / reps * 1e-3), "unit": "frames/s", "scaling": "strong"}
    steady = None
    if world == 1 and args.steady_steps > 0:
        # a long steady-state leg with its own clocks record (the driver's --steps 20 window is ~0.1 s)
        s2 = ClockSampler(local)
        s2.start()
        ms_long, _ = timed(step_device, args.steady_steps, 3, collective=False)
        steady = {"steps": args.steady_steps, "seconds": ms_long * 1e-3, "ms_per_step": ms_long / args.steady_steps,
                  "value": B * args.steady_steps / (ms_long * 1e-3), "unit": "frames/s", "clocks": s2.stop()}

    # ---- e2e through the reference-facing API, host in / host out -----------------------------
    h2d = B * 85 * 4
    d2h = B * 3 * size * size * 4
    pinned = [th.numpy().copy() for th in host_sets]

    # One call per timed region, as a user drives a whole motion sequence (run_imitator.py:224-241): steps x B frames go
    # through Imitator.inference_by_smpls in chunks of B; every chunk's SMPL vectors come from host memory and every
    # chunk's frames are copied back to pinned host memory inside the timed region (the D2H of chunk i overlaps the
    # compute of chunk i+1; the call returns only when every frame is on the host).
    def e2e_frames(nsteps, first):
        return [f for i in range(nsteps) for f in pinned[(first + i) % len(pinned)]]

    def run_e2e(nsteps, first, **kw):
        outs = imitator.inference_by_smpls(e2e_frames(nsteps, first), cam_strategy="smooth", **kw)
        assert len(outs) == nsteps * B
        return outs

    def timed_call(fn):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        t0 = time.time()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ms = max(e0.elapsed_time(e1), (time.time() - t0) * 1e3)        # the call is synchronous: host clock covers the D2H tail
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = t.item()
            dist.barrier()
        return ms
    # ---- HMR image encoder (frames driven from video, tgt_smpls=None): ms per frame at batch B, device-resident images
    hmr_leg = None
    if rank == 0 and not args.profile_range:
        full = dict(body.state_dict())
        full.update(S.synthetic_hmr_state(body.state_dict()))
        body.load_state_dict(full)
        body.eval()
        imgs = S.synthetic_hmr_inputs(B).to(dev)
        for _ in range(3):
            body(imgs)
        torch.cuda.synchronize()
        h0, h1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        h0.record()
        for _ in range(10):
            body(imgs)
        h1.record()
        torch.cuda.synchronize()
        hmr_leg = {"ms_per_frame": h0.elapsed_time(h1) / 10 / B, "batch": B,
                   "what": "HumanModelRecovery.forward (pre-activation ResNet-50 @224^2 on the conv engine + 3-iteration regressor); "
                           "added per frame when Imitator.inference is driven from images (tgt_smpls=None)"}
    # warm-up call = the same sequence (same first frame, hence the same 'smooth' cameras as the device-resident sets): the
    # pinned-host allocator is warm, the chunk graph captured, and a range-bit switch to fp16x3 -- a one-time event per
    # source and sequence -- has happened before the timed call, which then measures the steady state of the API
    run_e2e(max(args.steps, 3), 0)
    ms_e2e = timed_call(lambda: run_e2e(args.steps, 0))
    e2e_fps = world * B * args.steps / (ms_e2e * 1e-3)
    run_e2e(max(args.steps, 3), 0, as_uint8=True)
    ms_u8 = timed_call(lambda: run_e2e(args.steps, 0, as_uint8=True))
    h2d = B * 85 * 4
    d2h = B * 3 * size * size * 4

    line = {"metric": "frames/sec @256x256 (per-frame inference hot path)", "value": fps, "unit": "frames/s",
            "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": {"fp16f8": "f16 main product + e4m3 correction products (hi/lo split), f32 accumulate",
                      "fp16x3": "f16 (3-term hi/lo split, f32 accumulate)", "fp16": "f16, f32 accumulate"}[mode], "data": "synthetic",
            "config": workload_config(args),
            "e2e": {"value": e2e_fps, "unit": "frames/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": ms_e2e / args.steps,
                    "api": "ONE call Imitator.inference_by_smpls(steps x B host SMPL vectors) -> per chunk of B: H2D, SMPL LBS, raster, "
                           "generator, composite, D2H to pinned host (overlapping the next chunk) -> list of host float32 HxWx3 frames",
                    "hmr": hmr_leg,
                    "uint8_frames": {"value": world * B * args.steps / (ms_u8 * 1e-3), "unit": "frames/s",
                                     "d2h_bytes_per_step": B * 3 * size * size,
                                     "note": "same call with as_uint8=True: the BGR uint8 images the reference writes to disk"}},
            "precision": {"by_rank": modes_by_rank, "range_bits_rank0": policy_bits,
                          "policy": "default fp16f8; a rank whose frames raise a range bit (|x| >= 1024 or head pre-activations "
                                    "beyond +-8) runs fp16x3, exactly as Imitator.inference switches (LWB_AUTO_PRECISION)"},
            "gpu_launches": launches, "clocks": clocks, "steady_state": steady, "parity": parity, "config3_stream64": c3,
            "init_broadcast": {"bytes": bc_stats.get("bytes"), "ms": bc_stats.get("ms"),
                               "what": "the ONE collective: generator weights + source image, rank 0 -> all (NCCL), outside the timed region"},
            "personalize": {"ms_per_source": personalize_ms, "inpaintor_ms_per_source": inpaint_ms,
                            "what": "Imitator.personalize: SMPL LBS + raster + BG net + encode_src (host-synchronous wall clock, median of 5)"}}

    # ---- roofline of the conv engine + per-kernel-class breakdown (instrumented passes, rank 0) ---
    if rank == 0 and not args.no_extras:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        tf_peak = peaks.get("bf16_tflops_sustained") or 1400.0
        tf_burst = peaks.get("bf16_tflops") or 1650.0
        hbm_peak = peaks.get("hbm_gbs") or 6650.0
        src = "measured (MEASURED_PEAKS.json)" if peaks else "fallback (B200_PROFILING.md)"
        # per-kernel CUDA events need the kernels serialised (as ncu does): the instrumented passes run with LWB_STREAMS=1
        had_streams = os.environ.get("LWB_STREAMS")
        os.environ["LWB_STREAMS"] = "1"
        try:
            prof = GEN.profile_streams(lambda: [step_eager(i) for i in range(3)], lambda: [step_eager(i) for i in range(6)])
            ms_serial, _ = timed(step_eager, args.steps, 3, collective=False)
        finally:
            if had_streams is None:
                os.environ.pop("LWB_STREAMS", None)
            else:
                os.environ["LWB_STREAMS"] = had_streams
        line["streams"] = {"LWB_STREAMS": os.environ.get("LWB_STREAMS", "2 (default)"),
                           "cuda_graph": bool(captured is not None and captured.captured),
                           "ms_per_step_single_stream": ms_serial / args.steps,
                           "note": "roofline / breakdown / layers are measured with the kernels serialised (one stream), like ncu; "
                                   "value / e2e use LWB_STREAMS sub-batches whose kernels overlap"}
        conv = prof["conv"]
        issue_units = {"fp16x3": 3.0, "fp16f8": 2.0, "fp16": 1.0}[mode]
        ach = conv["flops"] / (conv["ms"] * 1e-3) / 1e12
        traffic, traffic_src = None, "absent"
        try:
            tj = json.load(open(os.path.join(ROOT, "profiles", "conv_traffic.json")))
            traffic, traffic_src = tj["bytes_per_launch"], tj.get("source", "round-1 capture")
        except Exception:
            pass
        line["roofline"] = {"bound": "tensor", "kernel": "k_conv_tc (tcgen05 implicit-GEMM, all conv layers of generator.inference)",
                            "achieved": ach, "peak": tf_peak, "unit": "TFLOP/s", "frac": ach / tf_peak, "traffic": traffic,
                            "peak_burst": tf_burst, "frac_vs_burst": ach / tf_burst,
                            "traffic_note": "mean DRAM bytes per conv launch from the committed ncu pass (profiles/conv_traffic.json: %s), "
                                            "not re-measured in this run" % traffic_src,
                            "peak_source": "bf16_tflops_sustained, " + src,
                            "algorithmic_gflop_per_step": conv["flops"] / prof["passes"] / 1e9,
                            "issued_mma_gflop_per_step": 3 * conv["flops"] / prof["passes"] / 1e9,
                            "issued_frac": issue_units * ach / tf_peak,
                            "issued_frac_note": "tensor-pipe time / elapsed: fp16x3 issues 3 fp16 products per algorithmic MAC; fp16f8 one "
                                                "fp16 product + two e4m3 products at twice the rate (assumed 2x the measured bf16 peak) = 2 units",
                            "ms_per_step_in_kernel": conv["ms"] / prof["passes"], "launches_per_step": conv["n"] / prof["passes"]}
        na = prof["norm"]
        line["roofline_hbm"] = {"bound": "hbm", "kernel": "k_norm_act (InstanceNorm+ReLU+residual+LWB warp-add)",
                                "achieved": na["bytes"] / (na["ms"] * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                                "frac": na["bytes"] / (na["ms"] * 1e-3) / 1e9 / hbm_peak,
                                "ms_per_step_in_kernel": na["ms"] / prof["passes"], "peak_source": "hbm_gbs, " + src}
        layers = {}
        for k, v in sorted(prof["layers"].items()):
            if k.startswith("conv/"):
                layers[k[5:]] = {"ms": round(v["ms"], 4), "n": v["n"], "tflops_algorithmic": round(v["work"] / (v["ms"] * 1e-3) / 1e12, 1)}
            elif k.startswith("heads/"):
                layers["heads " + k[6:]] = {"ms": round(v["ms"], 4), "n": v["n"], "tflops_algorithmic": round(v["work"] / (v["ms"] * 1e-3) / 1e12, 1)}
            elif k.startswith("norm/"):
                layers["norm " + k[5:]] = {"ms": round(v["ms"], 4), "n": v["n"], "gbs": round(v["work"] / (v["ms"] * 1e-3) / 1e9, 0)}
        line["layers"] = layers
        line["breakdown_ms_per_step"] = {k: prof[k]["ms"] / prof["passes"] for k in ("conv", "norm", "heads", "correspond", "input")}
        # the other precision modes of the conv engine, for transparency (the headline is the default mode)
        had = os.environ.get("LWB_PRECISION")
        pinned_mode = getattr(net, '_lwb_precision', None)
        net.set_precision(None)                                  # follow LWB_PRECISION for these legs (a policy switch pins the mode)
        try:
            modes, ref_pred = {}, None
            for m in ("fp16x3", "fp16f8", "fp16"):
                os.environ["LWB_PRECISION"] = m
                pred_m = step_eager(0).clone()
                if m == "fp16x3":
                    ref_pred = pred_m
                if m == mode:
                    fps_m = fps
                else:
                    ms_m, _ = timed(step_eager, args.steps, 3, collective=False)      # eager launches (no graph) for these legs
                    fps_m = world * B * args.steps / (ms_m * 1e-3)
                modes[m] = {"value": fps_m, "unit": "frames/s", "max_abs_vs_fp16x3": (pred_m - ref_pred).abs().max().item()}
            modes["fp16"]["note"] = "single-pass fp16: does not meet the 1e-3 parity bar; not the headline"
            line["precision_modes"] = modes
            line["fast_mode"] = dict(modes["fp16"], precision="single-pass fp16")
        finally:
            net.set_precision(pinned_mode)
            if had is None:
                os.environ.pop("LWB_PRECISION", None)
            else:
                os.environ["LWB_PRECISION"] = had
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline(size)
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()                      # the other ranks wait here while rank 0 finishes its (rank-local) extras
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
