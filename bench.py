#!/usr/bin/env python
"""Benchmark of the READ per-frame render hot path on B200 (driver contract: one JSON line on stdout).

    python bench.py --gpus 1 --steps K --warmup W [--config c1|c2|c3]   # our arm
    python bench.py --impl reference --gpus 1 ...                       # the reference's CPU path (oracle port) on host cores
    python bench.py ... --dump-outputs DIR                              # also write the last timed step's outputs as DIR/*.npy
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...

A "step" is one frame: clear + project/cull/z-resolve all points into the 4-level packed pyramid, gather the descriptor feature
pyramid, run the full 99-layer gated-conv refinement net -> RGB frame.  Workloads (BASELINE.json configs): c3 (default, the
config the metric is quoted on) = 10 M-point street scene at 1920x1080 (rendered 1920x1088 = padded to the %16 the net needs,
READ/gl/nn.py:107-109); c2 = 1 M points, 512x512; c1 = 100 k points, 256x256.
With N > 1 GPUs the cloud is sharded by spatial tile, every step renders N camera views together (one pass over each shard for all
views, ONE NCCL reduce-scatter(min) of the packed level-0 z-buffers so that rank r receives view r) and rank r refines view r
(frame-parallel net): N frames per step, weak scaling.

Output keys (DESIGN.md "Measurement"): value = frames/s with all inputs resident in HBM; e2e = frames/s through the public plugin
call (FrameRenderer.infer: host matrix inverse, H2D of the camera, D2H of the displayable frame, stream sync) - the headline;
roofline = the dominant kernel family (tcgen05 3x3 gated convs, tensor bound) measured live with CUDA events against the BURST
bf16 peak (launches timed in sequence, CUDA events between them); roofline_raster = rasterizer + gather against HBM bandwidth; parity = the timed frame
checked against the oracle (index maps bit-exact, RGB within the stated tolerance); cpu_baseline = the oracle port on the host
cores (one full frame); reference_gpu = the reference's own GPU path (its pcpr kernel + torch/cuDNN fp32 net) on this box.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

LEVELS = 4
CONFIGS = {
    # name: (points, width, rendered height, named height, scene depth, BASELINE.json description)
    "c3": (10_000_000, 1920, 1088, 1080, 250.0,
           "synthetic 10M-point street scene, 1920x1080 (rendered 1920x1088: padded to %16, crop), L=4 pyramid, descriptor dim 8, full MIMO-UNet refine"),
    "c2": (1_000_000, 512, 512, 512, 250.0, "kitti6-like synthetic street scene, 1M points, 512x512, L=4 pyramid, descriptor dim 8, full MIMO-UNet refine"),
    "c1": (100_000, 256, 256, 256, 60.0, "100k-point synthetic scene, 256x256, single view, L=4 pyramid, descriptor dim 8, full MIMO-UNet refine"),
}
C5 = dict(n_points=5_000_000, W=256, H=256, crops_per_gpu=8, depth=250.0,
          workload="train loop: 256x256 random crops (zoom U(0.7,2), shift), 5M points, batch 8 crops per GPU, L1 loss, "
                   "backward through gather + UNet, Adam (net) + RMSprop (descriptors)")
TOL_BF16, PSNR_BF16 = 3e-2, 45.0             # the stated production-mode tolerance (tests/test_gpu_unet.py, DESIGN.md §2)
DUMP_LIMIT_BYTES = 64 << 20


def metric_name(cfg):
    n, w, _, hn, _, _ = CONFIGS[cfg]
    return f"frames/sec @{w}x{hn}, {n // 1_000_000}M pts" if n >= 1_000_000 else f"frames/sec @{w}x{hn}, {n // 1000}k pts"


def measured_traffic():
    """DRAM bytes per launch from the committed ncu captures (profiles/r02_traffic.json, else r01); None if absent."""
    for name in ("r02_traffic.json", "r01_traffic.json"):
        p = os.path.join(ROOT, "profiles", name)
        try:
            d = json.load(open(p))
            d["_src"] = "profiles/" + name
            return d
        except Exception:
            continue
    return None


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"],
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "src": "MEASURED_PEAKS.json"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "src": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "50", "-i", str(index)], stdout=subprocess.PIPE,
                                      stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        try:
            out = self.p.communicate(timeout=5)[0]
        except Exception:
            out = ""
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[2:6]):
                if v == "Active":
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def dump_outputs(out_dir, arrays):
    """--dump-outputs: write each array (name -> numpy array) as out_dir/<name>.npy, float64 kept, everything else as float32,
    so that two builds run with the same arguments can be compared output for output."""
    arrays = {k: np.asarray(v) for k, v in arrays.items()}
    arrays = {k: a if a.dtype == np.float64 else a.astype(np.float32) for k, a in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit(f"bench.py --dump-outputs: {total} bytes of outputs exceed the {DUMP_LIMIT_BYTES} byte limit")
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


def psnr(a, b):
    peak = float(np.abs(b).max())
    mse = float(((a - b) ** 2).mean())
    return 99.0 if mse == 0 else float(10.0 * np.log10(peak * peak / mse))


# ---------------------------------------------------------------------------------------------- CPU arm
def host_threads():
    """Threads the CPU arm may use: affinity mask, capped by the cgroup CPU quota when there is one."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = max(1, min(n, int(float(q) / float(per) + 0.5)))
    except Exception:
        pass
    return n


def cpu_model():
    """'model name' of the host CPU (SURVEY.md §8d: print it next to the CPU timing)."""
    try:
        for line in open("/proc/cpuinfo"):
            if line.lower().startswith("model name"):
                return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def pick_torch_threads(sd):
    """torch's CPU convolutions do not scale to every core of a large shared host (oversubscription made a 128-thread
    run 25x slower than an 8-thread one): time one mid-size gated conv at a few thread counts and keep the fastest,
    so the CPU baseline is the best the host can do rather than an artefact."""
    import torch
    from oracle import unet_ref
    avail = host_threads()
    cands = sorted({c for c in (avail, 64, 32, 16, 8) if c <= avail})
    x = torch.rand(1, 64, 256, 512)
    best, best_t = cands[0], None
    for c in cands:
        torch.set_num_threads(c)
        with torch.no_grad():
            unet_ref.basic_conv(sd, "Encoder.1.layers.0.main.0", x, 3)
            t0 = time.perf_counter()
            for _ in range(3):
                unet_ref.basic_conv(sd, "Encoder.1.layers.0.main.0", x, 3)
            t = time.perf_counter() - t0
        if best_t is None or t < best_t:
            best, best_t = c, t
    torch.set_num_threads(best)
    return best, avail


def cpu_reference_frame(cfg, xyz, tex_cn, sd, pose=7):
    """ONE full frame of the reference's CPU path (oracle port), nothing extrapolated: sequential z-buffer of all 4 levels over
    all points (oracle/zbuffer.c, one host thread per level) + descriptor gather + the refinement net at the full rendered
    resolution (oracle/unet_ref.py, torch CPU fp32 on the chosen thread count).  Returns (seconds, info, index maps, RGB)."""
    import torch
    import oracle
    from oracle import unet_ref
    from read_b200 import synth
    _, W, H, _, _, _ = CONFIGS[cfg]
    proj, view = synth.camera_batch(W, H, [pose])
    t0 = time.perf_counter()
    _, idx, dep = oracle.render_pyramid(xyz, proj, view, W, H, LEVELS, threads=LEVELS)
    t_raster = time.perf_counter() - t0
    t0 = time.perf_counter()
    with torch.no_grad():
        feats = [unet_ref.point_texture(tex_cn, torch.from_numpy(idx[l])) for l in range(LEVELS)]
        out = unet_ref.unet_forward(sd, feats)
    t_net = time.perf_counter() - t0
    return t_raster + t_net, {"raster_s": t_raster, "gather_net_s": t_net}, (idx, dep), out


def scene_cpu(cfg):
    import torch
    from read_b200 import synth
    n, _, _, _, depth, _ = CONFIGS[cfg]
    xyz = synth.street_scene(n, depth=depth)
    tex = torch.rand((1, 8, n), generator=torch.Generator().manual_seed(synth.SEED))
    return xyz, tex


def base_config(cfg):
    n, W, H, _, _, desc = CONFIGS[cfg]
    return {"workload": desc, "config_id": cfg, "n_points": n, "width": W, "height": H, "levels": LEVELS}


def run_reference_arm(args):
    """The reference's own CPU implementation of the path (oracle port: the reference's GPU rasterizer has no CPU build and its
    Python modules cannot travel to the GPU box) on this box's host cores, full frames, same workload / config keys as our arm.
    --steps / --warmup are honoured up to a wall-clock budget (a C3 frame costs ~20 s of CPU time); the line says what ran."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import oracle
    from read_b200 import synth
    oracle.build()
    cfg = args.config
    sd = synth.synth_state_dict(synth.SEED)
    cores, avail = pick_torch_threads(sd)
    xyz, tex = scene_cpu(cfg)
    budget_s = float(os.environ.get("READ_BENCH_CPU_BUDGET_S", "900"))
    t_start = time.perf_counter()
    warm_done = 0
    for _ in range(args.warmup):
        if warm_done >= 1 and time.perf_counter() - t_start > 0.2 * budget_s:
            break
        cpu_reference_frame(cfg, xyz, tex, sd)
        warm_done += 1
    ts, info = [], None
    for _ in range(max(1, args.steps)):
        t, info, _, rgb = cpu_reference_frame(cfg, xyz, tex, sd)
        ts.append(t)
        if time.perf_counter() - t_start + t > budget_s:
            break
    steps = len(ts)
    t_total = float(np.sum(ts))
    fps = steps / t_total
    sample = (f"{steps} full frame(s) (requested {args.steps}, wall-clock budget {budget_s:.0f} s), {warm_done} warm-up: sequential z-buffer of all "
              f"{LEVELS} levels over {CONFIGS[cfg][0]} points (1 thread/level) + gather + full-resolution refinement net; torch threads "
              f"{cores} = fastest of a sweep up to the {avail} available; nothing extrapolated")
    line = {"impl": "reference", "metric": metric_name(cfg), "value": fps, "unit": "frames/s", "n_gpus": args.gpus,
            "steps": steps, "warmup": warm_done, "ms_per_step": t_total / steps * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": base_config(cfg),
            "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": cores, "cpu": cpu_model(), "kind": "port", "sample": sample,
                             "raster_s": info["raster_s"], "gather_net_s": info["gather_net_s"]},
            "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"rgb": rgb.numpy()})
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------- reference GPU path
def reference_gpu_block(cfg, xyz_np, tex_cn, sd, dev, frames=3):
    """What a READ user has on this box today (SURVEY §8d "kernel to beat"): the UNMODIFIED reference rasterizer (oracle/_ref,
    compiled from its own sources) called like src/READ/gl/myrender.py:32-40 - CPU tensors in, one pcpr.forward per level, CPU
    tensors out - followed by the reference's torch modules on the GPU in fp32 (oracle/unet_ref.py restates them op for op:
    index_select gather + cuDNN convs), with cuDNN's TF32 default and with TF32 off."""
    import torch
    from oracle import build_ref, unet_ref
    from read_b200 import synth
    pcpr = build_ref.load()
    if pcpr is None:
        return {"unavailable": "oracle/_ref/pcpr*.so not built (needs /root/reference at build time)"}
    _, W, H, _, _, _ = CONFIGS[cfg]
    pts = torch.from_numpy(xyz_np)
    sd_d = {k: v.to(dev) for k, v in sd.items()}
    tex_d = tex_cn.to(dev)
    sizes = [(int(W * 0.5 ** l), int(H * 0.5 ** l)) for l in range(LEVELS)]
    res = {}
    for tf32 in (True, False):
        torch.backends.cudnn.allow_tf32 = tf32
        torch.backends.cuda.matmul.allow_tf32 = tf32
        t_r, t_n = [], []
        for f in range(frames + 1):
            proj, view = synth.camera_batch(W, H, [7 + f])
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            total_m = torch.from_numpy(synth.total_matrix(proj, view))
            idx = [pcpr.forward(pts, total_m, w, h, 512)[0] for (w, h) in sizes]          # CPU in, CPU out, sync inside
            t1 = time.perf_counter()
            with torch.no_grad():
                out = unet_ref.net_and_texture(sd_d, tex_d, [i[:, None].to(dev) for i in idx])
            torch.cuda.synchronize()
            t2 = time.perf_counter()
            if f > 0:
                t_r.append(t1 - t0); t_n.append(t2 - t1)
        key = "tf32" if tf32 else "fp32"
        res[key] = {"raster_ms": float(np.median(t_r) * 1e3), "gather_net_ms": float(np.median(t_n) * 1e3),
                    "frames_per_s": float(1.0 / (np.median(t_r) + np.median(t_n)))}
    torch.backends.cudnn.allow_tf32 = True
    del sd_d, tex_d
    torch.cuda.empty_cache()
    res["how"] = (f"pcpr.forward(points_cpu, total_m_cpu, w, h, 512) x {LEVELS} levels (reference kernel, host<->device copies and device "
                  f"sync inside each call) + index maps to the GPU + PointTexture/UNet in torch fp32 eager (cuDNN); median of {frames} frames, wall clock")
    return res


# ---------------------------------------------------------------------------------------------- GPU arm
def run_ours(args):
    import torch
    import torch.distributed as dist
    from read_b200 import synth, ops, _lib as L, dist as rdist
    from read_b200.viewer import FrameRenderer

    cfg = args.config
    N_POINTS, W, H, H_NAMED, depth, _ = CONFIGS[cfg]
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.gpus != world:
        if world == 1 and args.gpus > 1:
            raise SystemExit("bench.py --gpus N>1 must be launched with torch.distributed.run (one rank per GPU)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"          # keep stdout to the one JSON line (NCCL prints its banner there)
        dist.init_process_group("nccl", device_id=dev)
    L.require_device(local)
    lib = L.load()
    if args.profile_timed_region and os.environ.get("READ_BENCH_PROFILE_PDL", "0") == "0":
        # ncu's graph-node profiling failed (LaunchFailed) on graphs with programmatic-dependency edges: the launch list is taken
        # with plain stream order (kernel durations are unaffected; ncu serialises the launches anyway)
        L.check(lib.read_set_option(b"tc_pdl", 0))
    pk = peaks()

    # ---- scene state (loaded once, like MyRender.update_ds / load_textures): resident in HBM.  The public plugin object owns it.
    xyz_np, tex_cpu = scene_cpu(cfg)
    sd = synth.synth_state_dict(synth.SEED)
    fr = FrameRenderer(xyz_np, sd, tex_cpu, (W, H), device=dev)
    fr.model.net.precision = args.precision
    net, tex = fr.model.net, fr.model._texture(0)
    start, count = rdist.shard_range(N_POINTS, rank, world)
    store = fr.store
    if world > 1:
        # rank r keeps the r-th contiguous range of the Morton order = a compact spatial tile of the scene
        sub = store.shard(start, count)
        sub.pts4, sub.perm = sub.pts4.clone(), sub.perm.clone()
        fr.store = store = sub
        fr.xyz = None
        torch.cuda.empty_cache()
    B = world                                   # views per step
    if args.profile_timed_region and os.environ.get("READ_BENCH_NO_GRAPH") == "1":
        net.use_graph = False                   # profiling aid: eager replay of the same launches
    eng = net.engine(1, H, W, dev)              # each rank refines ONE view per step
    tex_nd = tex.point_major()
    layout = L.FEAT_NHWC_BF16 if eng.bf16 else L.FEAT_NHWC_F32
    pyr = ops.Pyramid(B, W, H, LEVELS, dev)
    plane = W * H

    n_poses = 64
    total = args.warmup + args.steps + (1 if world > 1 else 0)     # N > 1: one extra camera set so that the LAST timed step also looks ahead
    pose_ts = [[(s * B + v) % n_poses for v in range(B)] for s in range(total)]
    cams = [synth.camera_batch(W, H, pose_ts[s]) for s in range(total)]          # host-side (proj, view) per step
    mats_host = torch.empty((total, B, 4, 4), dtype=torch.float32).pin_memory()
    for s in range(total):
        mats_host[s] = torch.from_numpy(synth.total_matrix(*cams[s]))
    mats_dev = mats_host.to(dev)
    frame_host = torch.empty((H, W, 4), dtype=torch.float32).pin_memory()
    frame_host_rgb = torch.empty((3, H, W), dtype=torch.float32).pin_memory()

    # N > 1: read_b200.dist.ShardedFrameStream - one pass over the shard for all views, ONE reduce-scatter (rank r gets view r), fused
    # resolve + gather, net; the rasterizer + collective of step s+1 run on a side stream under the net of step s
    sfs = rdist.ShardedFrameStream(store, tex_nd, eng, W, H, LEVELS, layout) if world > 1 else None

    def step(m_dev, m_next=None):
        """m_dev [B,4,4] on device -> eng.output [1,3,H,W] on device."""
        if world == 1:
            # level 0 is left cleared by the previous frame's fused resolve (reset_level0)
            ops.raster_project_sorted(pyr, store, m_dev)
            ops.pyramid_resolve_gather(tex_nd, pyr, eng.inputs, layout, reset_level0=True)
            return eng.run()
        return sfs.step(m_dev, m_next)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, first, finish=None):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for s in range(steps):
            fn(first + s)
        if finish is not None:
            finish()                         # e.g. join the copy stream: the last frame's D2H is inside the timed region
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    def resident_step(s):
        step(mats_dev[s], mats_dev[s + 1] if s + 1 < total else None)

    if world == 1:
        def e2e_step(s):
            # the plugin call a viewer makes (READ/gl/nn.py:113-129): host-side proj @ inv(view), H2D of the matrix, the whole
            # frame, the displayable [H,W,4] surface; then the frame goes to pinned host memory
            out = fr.infer(cams[s][0][0], cams[s][1][0])
            ready = torch.cuda.Event()
            ready.record()
            with torch.cuda.stream(copy_stream):                 # D2H of frame i on the copy engine while frame i+1 renders
                copy_stream.wait_event(ready)
                frame_hosts[s & 1].copy_(out['output'], non_blocking=True)
                out['output'].record_stream(copy_stream)
                copied[s & 1].record()
            if s >= 1:
                copied[(s - 1) & 1].synchronize()                # host side: the PREVIOUS frame is in host memory before we go on
        copy_stream = torch.cuda.Stream()
        frame_hosts = [frame_host, torch.empty_like(frame_host).pin_memory()]
        copied = [torch.cuda.Event(), torch.cuda.Event()]
        e2e_finish = lambda: torch.cuda.current_stream().wait_stream(copy_stream)
        e2e_h2d, e2e_d2h = 64, H * W * 4 * 4
        e2e_note = ("FrameRenderer.infer(proj, view) per step: host numpy proj @ inv(view), H2D of the 4x4 matrix through a pinned staging ring, raster + gather + "
                    "net + RGBA surface + net_input list, then D2H of the [H,W,4] f32 frame to pinned memory on a copy stream (double-buffered: the host "
                    "waits for frame i-1 while frame i renders; the last frame's copy is joined before the closing event); point cloud / "
                    "descriptors / weights are scene state resident in HBM (as MyRender.update_ds / load_textures)")
    else:
        e2e_next = {}

        def e2e_step(s):
            m = e2e_next.pop(s, None)
            if m is None:
                m = mats_host[s].to(dev, non_blocking=True)             # H2D of this step's cameras (pinned)
            mn = mats_host[s + 1].to(dev, non_blocking=True) if s + 1 < total else None      # ... and of the next step's (look-ahead)
            if mn is not None:
                e2e_next[s + 1] = mn
            out = step(m, mn)
            frame_host_rgb.copy_(out[0], non_blocking=True)              # D2H of the frame this rank produced
            torch.cuda.current_stream().synchronize()
        e2e_h2d, e2e_d2h = B * 64, 3 * H * W * 4
        e2e_note = ("distributed step per rank: pinned H2D of a step's B camera matrices (one step ahead), sharded raster + reduce-scatter of step "
                    "s+1 on a side stream under gather + net of step s, D2H of this rank's RGB frame to pinned memory, stream sync "
                    "(FrameRenderer is the single-GPU plugin object)")

    # ---- warm-up (also builds the CUDA graph)
    pyr.clear()
    for s in range(args.warmup):
        resident_step(s)
    torch.cuda.synchronize()
    launches_per_step = (2 + eng.n_launches()) if world == 1 else (4 + eng.n_launches())
    if args.profile_timed_region:
        # ncu --profile-from-start off: the capture holds exactly the launches of the timed steps (the launch list under profiles/);
        # numbers printed by such a run are not bench values, so nothing else is measured
        torch.cuda.synchronize()
        torch.cuda.cudart().cudaProfilerStart()
        ms_p = timed(resident_step, args.steps, args.warmup)
        torch.cuda.cudart().cudaProfilerStop()
        if rank == 0:
            print(json.dumps({"profiled_steps": args.steps, "launches_per_step": launches_per_step, "ms_under_profiler": ms_p,
                              "note": "profiling run: not a bench value"}))
        return
    sampler = ClockSampler(local) if rank == 0 else None
    join_side = (lambda: torch.cuda.current_stream().wait_stream(sfs.side)) if world > 1 else None   # K rasters inside K timed steps
    ms_res = timed(resident_step, args.steps, args.warmup, finish=join_side)
    clocks = sampler.stop() if sampler else None
    last_rgb = eng.output.clone() if args.dump_outputs and rank == 0 else None   # what step() returned last; the next run overwrites it
    if world == 1:
        pyr.clear()
    for s in range(min(3, args.warmup)):
        e2e_step(s)
    ms_e2e = timed(e2e_step, args.steps, args.warmup, finish=e2e_finish if world == 1 else join_side)
    fps = B * args.steps / (ms_res * 1e-3)
    fps_e2e = B * args.steps / (ms_e2e * 1e-3)

    # ---- live per-kernel measurements for the rooflines (CUDA events on the launching stream, eager launches, PDL off so that
    #      consecutive launches of one layer do not overlap)
    def time_call(fn, reps=5):
        torch.cuda.synchronize()
        ts = []
        for _ in range(reps):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); fn(); b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b))
        return float(np.mean(ts[1:]))

    sp = L.stream_ptr()
    L.check(lib.read_set_option(b"tc_pdl", 0))
    tc_ms = tc_flops = gen_ms = gen_flops = tcg_ms = tcg_flops = tco_ms = tco_flops = 0.0
    tc_classes = {}
    layer_rows = []
    aux_ms = 0.0
    # every launch of the net timed IN SEQUENCE: the frame's launch order replayed eagerly on the launching stream with an event
    # between consecutive launches (host enqueue runs ahead of the GPU, so an interval = one kernel + its launch gap, in the cache
    # state the real frame sees); median of 3 replays after one warm replay
    if hasattr(eng, "set_side_chain"):
        eng.set_side_chain(False)            # per-layer timing: one stream, full grids
    n_ops = len(eng.ops)
    seq = np.zeros((4, n_ops))
    for r_ in range(4):
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(n_ops + 1)]
        torch.cuda.synchronize()
        evs[0].record()
        for i_, ly in enumerate(eng.ops):
            eng.launch_op(ly, sp)
            evs[i_ + 1].record()
        torch.cuda.synchronize()
        seq[r_] = [evs[i_].elapsed_time(evs[i_ + 1]) for i_ in range(n_ops)]
    seq_ms = np.median(seq[1:], axis=0)
    for i_, ly in enumerate(eng.ops):
        t = float(seq_ms[i_])
        if ly.plan is None:
            aux_ms += t
            layer_rows.append({"name": ly.name, "impl": -1, "ms": t, "gflop": 0.0, "tflops": 0.0})
            continue
        layer_rows.append({"name": ly.name, "impl": int(ly.impl), "ms": t, "gflop": ly.flops / 1e9,
                           "tflops": ly.flops / (t * 1e-3) / 1e12})
        if ly.impl == L.CONV_TCGEN05 and ly.k == 3 and ly.stride == 1:
            tc_ms += t; tc_flops += ly.flops          # the tensor-bound instances: 3x3 stride-1 C->C convs
            if getattr(ly, "cin", None) == getattr(ly, "cout", -1) and ly.cin in (32, 64, 128, 256):
                c_ = tc_classes.setdefault(f"C{ly.cin}", [0, 0.0, 0.0])
                c_[0] += 1; c_[1] += t; c_[2] += ly.flops
        elif ly.impl == L.CONV_TCGEN05:
            tco_ms += t; tco_flops += ly.flops        # 1x1 / stride-2 / RAW-term launches: HBM- and latency-bound
        elif ly.impl == L.CONV_TCGEN05_GATHER:
            tcg_ms += t; tcg_flops += ly.flops
        else:
            gen_ms += t; gen_flops += ly.flops
    L.check(lib.read_set_option(b"tc_pdl", 1))
    m0 = mats_dev[args.warmup][:1].contiguous() if world == 1 else mats_dev[args.warmup]

    def project(m):
        ops.raster_project_sorted(pyr, store, m)

    def raster_frame():                      # what a frame does before the net (level 0 is clean on entry)
        project(m0)
        ops.pyramid_resolve_gather(tex_nd, pyr, eng.inputs, layout, view0=rank if world > 1 else 0,
                                   nviews=1 if world > 1 else None, reset_level0=(world == 1))
        if world > 1:
            L.check(lib.read_zbuf_clear(pyr.buf.data_ptr(), B * plane, sp))

    def one_shot(fn):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)

    pyr.clear()
    rg_ms = time_call(raster_frame, reps=6)
    project_ms, resolve_ms = [], []
    for _ in range(5):                       # the two halves separately (each on the state the other leaves behind)
        project_ms.append(one_shot(lambda: project(m0)))
        resolve_ms.append(one_shot(lambda: ops.pyramid_resolve_gather(tex_nd, pyr, eng.inputs, layout, view0=0, nviews=1,
                                                                      reset_level0=True)))
    project_ms, resolve_ms = float(np.mean(project_ms[1:])), float(np.mean(resolve_ms[1:]))
    if world > 1:
        pyr.clear()
    P = sum(w_l * h_l for (w_l, h_l) in pyr.sizes)
    feat_bytes = 2 if eng.bf16 else 4
    # algorithmic bytes (SURVEY.md §8d): xyz once (12 B/point) + per pyramid pixel: packed z write (8) + descriptor read (32) +
    # feature write (8 * s).  The packed z is counted ONCE.
    rg_bytes = 12 * count + P * (8 + 32 + 8 * feat_bytes)
    hbm = pk["hbm_gbs"]
    tens_peak = pk["bf16_tflops"]            # the conservative denominator: the burst peak, although the layers are timed in sequence
    roof_tc = None
    traf = measured_traffic()
    if tc_ms > 0:
        ach = tc_flops / (tc_ms * 1e-3) / 1e12
        kern = {"C32": "gated_conv_tc_kernel (one CTA, resident weights)", "C64": "gated_conv_tc2_kernel (CTA pair, resident weights)",
                "C128": "gated_conv_tc2s_kernel (CTA pair, streamed weights)", "C256": "gated_conv_tc2s_kernel (CTA pair, streamed weights)"}
        roof_tc = {"kernel": "tcgen05 implicit-GEMM gated conv, 3x3 stride-1 instances (gated_conv_tc_kernel / gated_conv_tc2_kernel / "
                             f"gated_conv_tc2s_kernel) = {100.0 * tc_flops / max(eng.flops, 1):.1f}% of the net's conv FLOPs", "bound": "tensor",
                   "by_class": {k_: {"layers": v_[0], "us_per_layer": 1e3 * v_[1] / v_[0], "tflops": v_[2] / (v_[1] * 1e-3) / 1e12,
                                     "frac": v_[2] / (v_[1] * 1e-3) / 1e12 / tens_peak, "kernel": kern[k_]} for k_, v_ in tc_classes.items()},
                   "achieved": ach, "peak": tens_peak, "unit": "TFLOP/s", "frac": ach / tens_peak,
                   "peak_src": pk["src"] + " bf16_tflops (burst figure; launches timed in sequence inside the eager replay of the net)",
                   "frac_of_sustained": ach / pk["bf16_tflops_sustained"], "sustained_peak": pk["bf16_tflops_sustained"],
                   "traffic": (traf or {}).get("gated_conv_tc_kernel_avg_bytes_per_launch"),
                   "traffic_src": (traf or {}).get("_src"),
                   "ms_per_frame": tc_ms,
                   "whole_net_tflops_in_graph": eng.flops / (ms_res / args.steps * 1e-3) / 1e12,
                   "layers": sum(1 for l_ in eng.layers if l_.impl == L.CONV_TCGEN05 and l_.k == 3 and l_.stride == 1)}
    ach_r = rg_bytes / (rg_ms * 1e-3) / 1e9
    roof_raster = {"kernel": "raster_stream_kernel + pyramid_resolve_gather_kernel",
                   "bound": "hbm",
                   "achieved": ach_r, "peak": hbm, "unit": "GB/s", "frac": ach_r / hbm, "peak_src": pk["src"],
                   "traffic": ((traf.get("raster_stream_kernel_bytes_per_launch", traf.get("raster_sorted_kernel_bytes_per_launch", 0))
                                + traf.get("pyramid_resolve_gather_bytes_per_launch", 0)) if traf else None),
                   "algorithmic_bytes": rg_bytes, "ms_per_frame": rg_ms,
                   "note": "algorithmic bytes = 12 B per point + 56 B per pyramid pixel (SURVEY 8d, bf16 features); the sorted store holds 16 B per point (xyz + original id)",
                   "project_ms": project_ms, "resolve_gather_ms": resolve_ms}
    gen_ach = gen_flops / (gen_ms * 1e-3) / 1e12 if gen_ms > 0 else None
    tcg_ach = tcg_flops / (tcg_ms * 1e-3) / 1e12 if tcg_ms > 0 else None

    # ---- latency mode (SURVEY.md §8f rank 1): all ranks cooperate on ONE frame - strip-parallel net with halo exchange over NVLink
    latency = None
    if world > 1:
        if H % (16 * world) != 0:
            latency = {"unavailable": f"frame height {H} is not a multiple of {16 * world}: strips need 16-row alignment per rank"}
        else:
            sf = rdist.StripFrameRenderer(store, tex_nd, sd, W, H, dev)
            m1 = mats_dev[args.warmup][:1].contiguous()
            for _ in range(3):
                got = sf.render(m1)
            for l in range(LEVELS):                      # the same feature pyramid through this rank's full-frame engine
                eng.inputs[l].copy_(sf.full_feats[l])
            same = torch.tensor([1 if torch.equal(got, eng.run()[0]) else 0], device=dev)
            dist.all_reduce(same, op=dist.ReduceOp.MIN)
            ms_lat = timed(lambda s_: sf.render(m1), args.steps, 0)
            latency = {"ms_per_frame": ms_lat / args.steps, "frames_per_s": args.steps / (ms_lat * 1e-3),
                       "frame_parallel_ms_per_frame": ms_res / args.steps,
                       "halo_exchanges_per_frame": sf.eng.n_exchanges(), "launches_per_frame": sf.eng.n_launches() + 3,
                       "bit_identical_to_single_gpu_net": bool(same.item()),
                       "how": "one view per step: sharded raster + NCCL all-reduce(min) of level 0 + gather on every rank, then each rank refines "
                              "its horizontal strip (halo rows through peer-mapped mailboxes, csrc/halo.cu) and the strips are all-gathered; "
                              "max over ranks, CUDA events"}
            del sf
            pyr.clear()
    if rank == 0 and args.layer_times:
        os.makedirs(os.path.dirname(os.path.abspath(args.layer_times)), exist_ok=True)
        json.dump(layer_rows, open(args.layer_times, "w"), indent=0)
    parity = None
    cpu_line = None
    ref_gpu = None
    if rank == 0 and world == 1:
        # ---- parity of the benchmarked configuration itself (VERDICT r01 #1): the frame of pose 7
        pose = 7
        proj, view = synth.camera_batch(W, H, [pose])
        mp = torch.from_numpy(synth.total_matrix(proj, view)).to(dev)
        pyr.clear()
        ops.raster_project_sorted(pyr, store, mp)
        ops.raster_derive(pyr)
        maps = [ops.zbuf_resolve(pyr, l) for l in range(LEVELS)]
        pyr.clear()
        gpu_rgb = fr.model.render(store, mp, W, H).cpu().numpy()
        parity = {"pose": pose, "tolerance": {"max_abs": TOL_BF16, "psnr_db": PSNR_BF16}}
        # (a) the bf16 tensor-core frame vs the fp32 CUDA-core engine on the identical feature pyramid
        from read_b200.engine import UNetEngine
        eng32 = UNetEngine(sd, 1, H, W, dev, precision="fp32", use_graph=False)
        ops.raster_project_sorted(pyr, store, mp)
        ops.pyramid_resolve_gather(tex_nd, pyr, eng32.inputs, L.FEAT_NHWC_F32, reset_level0=True)
        rgb32 = eng32.run().cpu().numpy()
        del eng32
        torch.cuda.empty_cache()
        parity["vs_fp32_engine"] = {"max_abs": float(np.abs(gpu_rgb - rgb32).max()), "psnr_db": psnr(gpu_rgb, rgb32)}
        ok = parity["vs_fp32_engine"]["max_abs"] < TOL_BF16 and parity["vs_fp32_engine"]["psnr_db"] > PSNR_BF16
        if not args.no_cpu_baseline:
            import oracle
            oracle.build()
            cores, avail = pick_torch_threads(sd)
            t_frame, info, (oidx, odep), cpu_rgb = cpu_reference_frame(cfg, xyz_np, tex_cpu, sd, pose)
            cpu_line = {"value": 1.0 / t_frame, "unit": "frames/s", "cores": cores, "cpu": cpu_model(), "kind": "port",
                        "sample": (f"1 full frame of this workload, nothing extrapolated: sequential z-buffer (4 levels, {N_POINTS} pts, 1 thread/level) = "
                                   f"{info['raster_s']:.2f} s + gather + refinement net at {W}x{H} = {info['gather_net_s']:.2f} s; "
                                   f"torch threads {cores} (fastest of a sweep, {avail} available)")}
            idx_eq = all(np.array_equal(maps[l][0].cpu().numpy(), oidx[l][:, 0]) for l in range(LEVELS))
            dep_eq = all(np.array_equal(maps[l][1].cpu().numpy().view(np.uint32), odep[l][:, 0].view(np.uint32)) for l in range(LEVELS))
            cpu_np = cpu_rgb.numpy()
            parity["vs_cpu_oracle"] = {"index_equal": bool(idx_eq), "depth_bits_equal": bool(dep_eq),
                                       "rgb_max_abs": float(np.abs(gpu_rgb - cpu_np).max()), "rgb_psnr_db": psnr(gpu_rgb, cpu_np),
                                       "rgb_fp32_engine_max_abs": float(np.abs(rgb32 - cpu_np).max())}
            ok = ok and idx_eq and dep_eq and parity["vs_cpu_oracle"]["rgb_max_abs"] < TOL_BF16 and parity["vs_cpu_oracle"]["rgb_psnr_db"] > PSNR_BF16
        parity["ok"] = bool(ok)
        if not args.no_reference_gpu:
            try:
                ref_gpu = reference_gpu_block(cfg, xyz_np, tex_cpu, sd, dev)
                if "tf32" in ref_gpu:
                    ref_gpu["our_e2e_speedup_vs_tf32"] = fps_e2e / ref_gpu["tf32"]["frames_per_s"]
                    ref_gpu["our_e2e_speedup_vs_fp32"] = fps_e2e / ref_gpu["fp32"]["frames_per_s"]
            except Exception as e:                      # the comparator must never take the bench line down
                ref_gpu = {"unavailable": f"{type(e).__name__}: {e}"[:300]}
    # ---- the reference-shaped surface (VERDICT r01 missing #6): what train.py / viewer.py call when they are NOT ported to the
    #      fused render(): MyRender.render(data) -> index maps on the host (myrender.py:12-43), then model(inputs dict)
    #      (NetAndTexture.forward, compose.py:125-181) with the maps moved to the GPU - same frame, same kernels underneath.
    surface = None
    if world == 1 and rank == 0:
        try:
            from read_b200.myrender import MyRender

            class _DS:
                pass
            ds = _DS()
            ds.id, ds.tgt_sh = 0, np.array([W, H])
            ds.input_format = ", ".join(["uv_1d_p1"] + [f"uv_1d_p1_ds{l}" for l in range(1, LEVELS)])
            ds.scene_data = {"pointcloud": {"xyz": xyz_np}}
            mr = MyRender([ds])
            ts_r, ts_m = [], []
            for s_ in range(4):
                proj_, view_ = cams[args.warmup + s_]
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                out_d, _ = mr.render({"input": {"id": torch.tensor([0])}, "proj_matrix": torch.from_numpy(proj_[:1]),
                                      "view_matrix": torch.from_numpy(view_[:1])})
                torch.cuda.synchronize()
                t1 = time.perf_counter()
                with torch.no_grad():
                    inp = {k: (v.to(dev) if torch.is_tensor(v) else v) for k, v in out_d.items()}
                    o_ = fr.model(inp)
                    o_ = o_["im_out"] if isinstance(o_, dict) else o_
                    _ = o_.float().mean().item()
                t2 = time.perf_counter()
                ts_r.append(t1 - t0); ts_m.append(t2 - t1)
            surface = {"myrender_render_ms": 1e3 * float(np.median(ts_r[1:])), "model_forward_ms": 1e3 * float(np.median(ts_m[1:])),
                       "frames_per_s": 1.0 / float(np.median(ts_r[1:]) + np.median(ts_m[1:])),
                       "how": "MyRender.render (unsorted cloud, index + depth maps returned as CPU tensors like the reference) + "
                              "NetAndTexture.forward(inputs dict) with the maps copied to the GPU; wall clock, median of 3 frames"}
            del mr
        except Exception as e:
            surface = {"unavailable": f"{type(e).__name__}: {e}"[:300]}
    if rank == 0:
        line = {
            "metric": metric_name(cfg), "value": fps, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_res / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16" if eng.bf16 else "f32", "data": "synthetic",
            "config": dict(base_config(cfg), views_per_step=B,
                           parallelism=(f"spatial-tile point shards x{world} (Morton ranges), all views in one pass per shard + one NCCL "
                                        f"reduce-scatter(min) + frame-parallel net") if world > 1 else "single GPU",
                           l2=("inputs larger than L2 (120 MB cloud, 16.7 MB z-buffer, >130 MB activations per layer at full res)" if cfg == "c3" else
                               "small workload: activations of the coarse layers fit L2; successive frames use different camera poses and every "
                               "layer writes its own buffer (6.6 GB of activations are touched per frame at c3; scaled by pixels here)"),
                           cuda_graph=bool(eng.use_graph), conv_impl=eng.impl_histogram()),
            "e2e": {"value": fps_e2e, "unit": "frames/s", "h2d_bytes_per_step": int(e2e_h2d),
                    "d2h_bytes_per_step": int(e2e_d2h), "ms_per_step": ms_e2e / args.steps, "note": e2e_note},
            "gpu_launches": int(launches_per_step * args.steps),
            "clocks": clocks,
            "roofline": roof_tc if roof_tc else roof_raster,
            "roofline_raster": roof_raster,
            "breakdown_ms_per_frame": {"raster_project": project_ms, "pyramid_resolve_gather": resolve_ms, "raster_total": rg_ms,
                                       "conv_tcgen05_tma_3x3": tc_ms, "conv_tcgen05_tma_other": tco_ms,
                                       "conv_tcgen05_tma_other_tflops": (tco_flops / (tco_ms * 1e-3) / 1e12 if tco_ms > 0 else None),
                                       "conv_tcgen05_gather": tcg_ms,
                                       "conv_tcgen05_gather_tflops": tcg_ach, "conv_generic": gen_ms, "upsample_kernels": aux_ms,
                                       "conv_generic_tflops": gen_ach, "net_flops": eng.flops,
                                       "note": "eager launches timed in sequence with CUDA events between them (PDL off); the frame replays them as one CUDA graph with PDL"},
            "parity": parity,
            "latency_mode": latency,
            "cpu_baseline": cpu_line,
            "reference_gpu": ref_gpu,
            "reference_surface": surface,
        }
        if last_rgb is not None:
            dump_outputs(args.dump_outputs, {"rgb": last_rgb.cpu().numpy()})
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
    if parity is not None and not parity["ok"]:
        sys.stderr.write("bench.py: PARITY FAILURE at the benchmarked configuration: " + json.dumps(parity) + "\n")
        sys.exit(1)



# ---------------------------------------------------------------------------------------------- training step (config c5)
def run_train(args):
    """BASELINE config 5: one optimisation step per "step" (src/train.py:257-266): rasterize the batch's crops, sample descriptors,
    refinement net forward + L1 loss + backward, data-parallel gradient join, Adam on the net and RMSprop on the descriptors.
    Ours: rasterizer (all crops in one pass), descriptor gather forward / sparse backward, sparse RMSprop, sparse gradient
    exchange.  Library (torch / cuDNN, stated in the line): the net's forward / backward in training mode, Adam, NCCL."""
    import torch
    import torch.distributed as dist
    from read_b200 import synth, ops, _lib as L, dist as rdist, train as rtrain
    from read_b200.unet import UNet
    from read_b200.texture import PointTexture
    from read_b200.compose import NetAndTexture
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"
        dist.init_process_group("nccl", device_id=dev)
    L.require_device(local)
    N, W, H, Bc = C5["n_points"], C5["W"], C5["H"], C5["crops_per_gpu"]
    xyz = torch.from_numpy(synth.street_scene(N, depth=C5["depth"])).to(dev)
    store = ops.SortedPoints(xyz)                          # every rank holds the scene; crops differ per rank (data parallel)
    tex = PointTexture(8, N, init_method='zeros')
    with torch.no_grad():
        tex.texture_.copy_(torch.rand((1, 8, N), generator=torch.Generator().manual_seed(synth.SEED)))
    net = UNet()
    net.load_state_dict(synth.synth_state_dict(synth.SEED), strict=True)
    model = NetAndTexture(net, {0: tex}, 1)
    model.load_textures(0)
    model.to(dev).eval()                                   # eval_in_train: BatchNorm uses running statistics (train.py:271-273)
    opt_net = torch.optim.Adam(net.parameters(), lr=1e-4)
    opt_tex = rtrain.SparseRMSprop(tex, lr=1e-1)
    net_params = [p for p in net.parameters()]
    pyr = ops.Pyramid(Bc, W, H, LEVELS, dev)
    total = args.warmup + args.steps
    rng = np.random.default_rng(synth.SEED + rank)
    mats_host = torch.empty((total, Bc, 4, 4), dtype=torch.float32).pin_memory()
    for s in range(total):
        ts = rng.integers(0, 64, Bc)
        mats_host[s] = torch.from_numpy(synth.total_matrix(*synth.crop_cameras(W, H, ts, rng)))
    mats_dev = mats_host.to(dev)
    target = torch.rand((Bc, 3, H, W), generator=torch.Generator().manual_seed(7 + rank)).to(dev)
    keys = ["uv_1d_p1"] + [f"uv_1d_p1_ds{l}" for l in range(1, LEVELS)]
    ids0 = torch.zeros(Bc, dtype=torch.long)
    tim = {"raster": 0.0, "net_fwd_bwd": 0.0, "join": 0.0, "optim": 0.0}
    ev = lambda: torch.cuda.Event(enable_timing=True)
    marks = []
    last = [None, None]

    def step(m_dev, profile=False):
        e = [ev() for _ in range(5)] if profile else None
        if profile: e[0].record()
        pyr.clear()
        ops.raster_project_sorted(pyr, store, m_dev)
        ops.raster_derive(pyr)
        inputs = {k: ops.zbuf_resolve(pyr, l, want_depth=False)[0].unsqueeze(1) for l, k in enumerate(keys)}
        inputs["id"] = ids0
        if profile: e[1].record()
        out = model(inputs)
        loss = torch.nn.functional.l1_loss(out, target) / world
        loss.backward()
        if profile: e[2].record()
        if world > 1:
            grads = [p.grad for p in net_params if p.grad is not None]
            flat = torch._utils._flatten_dense_tensors(grads)
            dist.all_reduce(flat)
            for g, f in zip(grads, torch._utils._unflatten_dense_tensors(flat, grads)):
                g.copy_(f)
            rtrain.exchange_sparse_grads(tex)
        if profile: e[3].record()
        opt_net.step()
        opt_tex.step()
        opt_net.zero_grad(set_to_none=True)
        if profile:
            e[4].record()
            marks.append(e)
        last[:] = [loss, out]
        return loss

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn):
        barrier()
        e0, e1 = ev(), ev()
        e0.record()
        for s in range(args.steps):
            fn(args.warmup + s)
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    for s in range(args.warmup):
        step(mats_dev[s])
    torch.cuda.synchronize()
    launches0 = ops.launch_count()
    sampler = ClockSampler(local) if rank == 0 else None
    ms_res = timed(lambda s: step(mats_dev[s]))
    clocks = sampler.stop() if sampler else None
    last_out = [t.detach().clone() for t in last] if args.dump_outputs and rank == 0 else None
    our_launches = ops.launch_count() - launches0

    def e2e_step(s):
        m = mats_host[s].to(dev, non_blocking=True)
        loss = step(m)
        return float(loss.item())                       # the loss is read back every step, as train.py logs it
    ms_e2e = timed(e2e_step)
    for s in range(3):
        step(mats_dev[args.warmup + s], profile=True)
    torch.cuda.synchronize()
    for e in marks:
        tim["raster"] += e[0].elapsed_time(e[1]) / len(marks)
        tim["net_fwd_bwd"] += e[1].elapsed_time(e[2]) / len(marks)
        tim["join"] += e[2].elapsed_time(e[3]) / len(marks)
        tim["optim"] += e[3].elapsed_time(e[4]) / len(marks)
    # the descriptor optimizer alone: ours (sparse) vs the reference's dense torch.optim.RMSprop on the same parameter
    step(mats_dev[0]); torch.cuda.synchronize()
    touched = None
    out = model({**{k: ops.zbuf_resolve(pyr, l, want_depth=False)[0].unsqueeze(1) for l, k in enumerate(keys)}, "id": ids0})
    torch.nn.functional.l1_loss(out, target).backward()
    touched = rtrain.touched_count(tex)
    a, b = ev(), ev()
    a.record(); opt_tex.step(); b.record(); torch.cuda.synchronize()
    sparse_ms = a.elapsed_time(b)
    opt_net.zero_grad(set_to_none=True)
    dense_p = torch.nn.Parameter(tex.texture_.detach().clone())
    dense_opt = torch.optim.RMSprop([dense_p], lr=0.1)
    dense_p.grad = torch.zeros_like(dense_p)
    dense_opt.step(); torch.cuda.synchronize()
    a, b = ev(), ev()
    a.record(); dense_opt.step(); b.record(); torch.cuda.synchronize()
    dense_ms = a.elapsed_time(b)
    pk = peaks()
    alg = N + touched * 8 * 4 * 7                        # flags + per touched element: grad r/w, square_avg r/w, param r/w, shadow w
    crops = world * Bc * args.steps
    if rank == 0:
        line = {"metric": "train crops/sec (256x256 crops, 5M pts)", "value": crops / (ms_res * 1e-3), "unit": "crops/s", "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_res / args.steps, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32 (net training in torch/cuDNN fp32; descriptors f32)", "data": "synthetic",
                "config": {"workload": C5["workload"], "config_id": "c5", "n_points": N, "width": W, "height": H, "levels": LEVELS,
                           "crops_per_gpu": Bc, "global_batch": world * Bc,
                           "parallelism": f"data parallel x{world}: NCCL all-reduce of the net's gradients (one flat bucket) + all-gather of the touched (id, grad[8]) descriptor rows" if world > 1 else "single GPU",
                           "ours": "rasterizer (all crops in one pass), index maps, descriptor gather forward, sparse gather backward, sparse RMSprop, sparse gradient exchange",
                           "library": "UNet forward/backward in training mode (torch operators, cuDNN), Adam, NCCL"},
                "e2e": {"value": crops / (ms_e2e * 1e-3), "unit": "crops/s", "h2d_bytes_per_step": Bc * 64, "d2h_bytes_per_step": 4,
                        "ms_per_step": ms_e2e / args.steps, "note": "crop cameras from pinned host memory every step, loss scalar read back every step"},
                "gpu_launches": int(our_launches),
                "clocks": clocks,
                "roofline": {"kernel": "sparse_rmsprop_kernel (descriptor optimizer, touched points only)", "bound": "hbm",
                             "achieved": alg / (sparse_ms * 1e-3) / 1e9, "peak": pk["hbm_gbs"], "unit": "GB/s",
                             "frac": alg / (sparse_ms * 1e-3) / 1e9 / pk["hbm_gbs"], "traffic": None, "algorithmic_bytes": alg,
                             "touched_points": touched, "ms": sparse_ms, "dense_torch_rmsprop_ms": dense_ms,
                             "note": "latency-bound at this size (a few 10^5 touched rows); the comparison that matters is the dense optimizer's time"},
                "breakdown_ms_per_step": tim,
                "cpu_baseline": None}
        if last_out is not None:
            dump_outputs(args.dump_outputs, {"loss": last_out[0].double().cpu().numpy(), "rgb": last_out[1].cpu().numpy()})
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="c3", choices=sorted(CONFIGS) + ["c5"])
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-reference-gpu", action="store_true")
    ap.add_argument("--profile-timed-region", action="store_true",
                    help="cudaProfilerStart/Stop around the timed steps and exit (for ncu --profile-from-start off)")
    ap.add_argument("--layer-times", default=None, help="write per-layer CUDA-event timings (JSON) to this path")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="after the timed steps, write what the last timed step computed as DIR/<name>.npy (rank 0's frame 'rgb' "
                         "[1,3,H,W]; c5: the step's 'loss' and its rendered crops 'rgb' [B,3,H,W])")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.config == "c5":
        if args.impl == "reference":
            print(json.dumps({"impl": "reference", "unavailable": "config c5 (training) has no CPU arm: the reference's training step needs its CUDA rasterizer"}))
        else:
            run_train(args)
    elif args.impl == "reference":
        run_reference_arm(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
