#!/usr/bin/env python
"""bench.py -- rays/sec of the NeO-360 ray-marching hot path on B200 (BASELINE.json metric).

Workload (BASELINE.json configs[1]): NeO-360 tri-planar render, 3 source views, 640x480 target frame,
128 coarse + 64 fine samples per ray and branch (129 + 193 points, fg and bg => 644 field evaluations per ray,
each over 3 views), chunk=1024 semantics (quirk Q1), synthetic NERDS360-shaped scene (neo360_b200/synth.py).
One "step" = one full frame (307 200 rays) through the hot path.  N GPUs: every rank renders its own frame of the
turntable (weak scaling, no data-path collective), value = all rays of all ranks / max-over-ranks device time.

  python bench.py [--gpus N] [--steps K] [--warmup W]            our CUDA path
  python bench.py --impl reference [...]                         the reference algorithm (CPU oracle port) on host cores
  python bench.py [...] --dump-outputs DIR                        also writes what the last timed step rendered as DIR/<name>.npy

Prints ONE JSON line (rank 0).  See the prompt contract for the keys; `roofline` is for the dominant kernel (the
field kernel: lookups + MLP), `cpu_baseline` is the oracle port timed on this box's host cores on a bounded sample.
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

IMG_W, IMG_H = 640, 480
N_COARSE, N_FINE, NV, CHUNK = 128, 64, 3, 1024
# reference-formulation MACs per (point, all 3 views): SURVEY.md section 8(a) a10
FLOP_PER_POINT = {0: 2 * 770688, 1: 2 * 786816}          # fg, bg
POINTS_PER_RAY = (N_COARSE + 1) + (N_COARSE + 1 + N_FINE)  # per branch
FLOP_PER_RAY = POINTS_PER_RAY * (FLOP_PER_POINT[0] + FLOP_PER_POINT[1])   # 1.003 GFLOP
# MACs the TC path actually needs per point (mean of fg/bg): per view the re-associated trunk 128*(KE+128+128+128+KE), the bilinear
# blend of the 4 maps (16 taps x 256 projected channels, on the tensor pipe since round 2) and the folded head 80*128; once per
# point the direction / colour head 80*32 + 64*64 + 16*64.  Padding of the tcgen05 tiles (window slots without a tap, K 63->64) is
# NOT counted: this is the useful work the tensor pipe has to do, the denominator of the honest roofline fraction.
ISSUED_MAC_PER_POINT = 0.5 * sum(3 * (128 * (2 * ke + 384) + 16 * 256 + 80 * 128) + 80 * 32 + 64 * 64 + 16 * 64 for ke in (64, 96))


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "eager-gpu"])
    ap.add_argument("--precision", default=os.environ.get("NEO360_PRECISION", "tc"), choices=["tc", "fp32"])
    ap.add_argument("--rays", type=int, default=IMG_W * IMG_H, help="debug only: fewer rays per step (not a valid headline)")
    ap.add_argument("--cpu-sample-rays", type=int, default=1024)
    ap.add_argument("--no-cpu-baseline", action="store_true", help="debug: skip the CPU oracle leg (and with it the parity block)")
    ap.add_argument("--no-extras", action="store_true", help="debug: skip the eager-GPU reference leg and the call-pattern variants")
    ap.add_argument("--mode", default="frames", choices=["frames", "strong", "turntable", "train", "mip360", "vanilla", "encoder"],
                    help="frames: BASELINE configs[1], one frame per rank (the headline, default); strong: ONE 640x480 frame split over the ranks "
                         "+ NCCL all-gather of the pixels (models/interface.py:30-50); turntable: BASELINE configs[4], views sharded first; "
                         "train: BASELINE configs[3], 4096-ray batches with an NCCL gradient all-reduce; mip360: BASELINE configs[2], "
                         "Mip-NeRF 360 at 640x480 with 64+64+64 samples, every dense layer on tcgen05")
    ap.add_argument("--views", type=int, default=100, help="turntable mode: number of target views")
    ap.add_argument("--batch-rays", type=int, default=4096, help="train mode: rays per optimisation step over all ranks")
    ap.add_argument("--train-matmul", choices=("fp32", "tf32"), default="fp32",
                    help="train mode: precision of the framework GEMMs of the dense layers.  tf32 = torch.backends.cuda.matmul.allow_tf32, the setting "
                         "the reference was trained under (torch 1.11 default, SURVEY.md 8(d))")
    ap.add_argument("--train-formulation", choices=("projected", "reference"), default="projected",
                    help="train mode: projected = map columns of layers 0/3 applied to the feature maps once per step (exact re-association, default); "
                         "reference = the reference's row-by-row K=703/831 input layers")
    ap.add_argument("--freeze-encoder", action="store_true", help="train mode: MLPs only (finetune mode); default trains GridEncoder inside the step")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned (render_rays_test's dict, rank 0) as DIR/<name>.npy, float32; the inputs "
                         "depend only on the arguments, so two builds can be compared output for output")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.mode != "frames"):
        ap.error("--dump-outputs needs --impl ours --mode frames")
    return args


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"bf16_tflops": d["bf16_tflops_sustained"], "burst": d["bf16_tflops"], "hbm_gbs": d["hbm_gbs"], "src": "measured (MEASURED_PEAKS.json, sustained)"}
    return {"bf16_tflops": 1400.0, "burst": 1590.0, "hbm_gbs": 6650.0, "src": "fallback (B200_PROFILING.md)"}


class ClockSampler(threading.Thread):
    """Samples SM clocks / throttle reasons through NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.samples, self.reasons, self.max_mhz = index, False, [], set(), None

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            names = {"hw_slowdown": 0x8, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40,
                     "sw_power_cap": 0x4, "hw_power_brake_slowdown": 0x80}
            while not self.stop_flag:
                self.samples.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
                time.sleep(0.05)
        except Exception as e:  # NVML missing: report that rather than inventing clocks
            self.reasons.add("nvml_unavailable:" + type(e).__name__)

    def result(self):
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


def build_scene_cpu():
    from neo360_b200 import synth
    sc = synth.make_scene((IMG_W, IMG_H), NV, (120, 160), seed=0)
    P = synth.make_mlp_params(0)
    return sc, P


def frame_rays_cpu(view):
    """Host-side ray generation for frame `view` of the 100-view turntable (datasets/ray_utils.py:84-176 semantics)."""
    import torch
    from neo360_b200 import synth
    pose = synth.target_pose(view, 100)
    j, i = torch.meshgrid(torch.arange(IMG_H, dtype=torch.float32), torch.arange(IMG_W, dtype=torch.float32), indexing="ij")
    f = 0.8 * IMG_W
    dirs = torch.stack([(i - IMG_W / 2) / f, -(j - IMG_H / 2) / f, -torch.ones_like(i)], -1)
    d = dirs @ pose[:3, :3].T
    d = (d / d.norm(dim=-1, keepdim=True)).reshape(-1, 3)
    o = pose[:3, 3].expand(d.shape).contiguous()
    return o, d


def cpu_reference_rate(sc, P, n_rays, steps=1, warmup=0, threads=None):
    """The reference's algorithm (oracle port, F.grid_sample lookups, eager torch CPU) on `n_rays` rays of frame 0,
    chunk = 1024 as the reference's render loop; encoder hoisted.  Returns (rays/s, seconds per step list)."""
    import torch
    from oracle import neo360_oracle as orc
    if threads is None:
        # eager torch on very wide hosts can be slower with every core than with a few dozen: probe and keep the best
        threads = os.cpu_count()
        if threads > 32:
            best = None
            o, d = frame_rays_cpu(0)
            for cand in (threads, 64, 32, 16):
                if cand > os.cpu_count():
                    continue
                torch.set_num_threads(cand)
                rr = {"rays_o": o[:128].contiguous(), "rays_d": d[:128].contiguous(), "viewdirs": d[:128].contiguous()}
                osc0 = orc.Scene(sc["planes_xz"], sc["planes_xy"], sc["planes_yz"], sc["latent"], sc["src_poses"],
                                 float(sc["src_focal"][0]), float(sc["src_c"][0, 0]), float(sc["src_c"][0, 1]), IMG_W, IMG_H)
                with torch.no_grad():
                    t0 = time.perf_counter()
                    orc.render_chunked(rr, osc0, P, N_COARSE, N_FINE, chunk=CHUNK, lookup_impl="aten")
                    dt = time.perf_counter() - t0
                if best is None or dt < best[0]:
                    best = (dt, cand)
            threads = best[1]
    torch.set_num_threads(threads)
    osc = orc.Scene(sc["planes_xz"], sc["planes_xy"], sc["planes_yz"], sc["latent"], sc["src_poses"],
                    float(sc["src_focal"][0]), float(sc["src_c"][0, 0]), float(sc["src_c"][0, 1]), IMG_W, IMG_H)
    o, d = frame_rays_cpu(0)
    start = (IMG_H // 2) * IMG_W
    rays = {"rays_o": o[start:start + n_rays].contiguous(), "rays_d": d[start:start + n_rays].contiguous(),
            "viewdirs": d[start:start + n_rays].contiguous()}
    times = []
    with torch.no_grad():
        for it in range(warmup + steps):
            t0 = time.perf_counter()
            out = orc.render_chunked(rays, osc, P, N_COARSE, N_FINE, chunk=CHUNK, lookup_impl="aten")
            dt = time.perf_counter() - t0
            if it >= warmup:
                times.append(dt)
    cpu_reference_rate.last = (rays, out)          # the oracle's pixels of the sample: bench's parity block compares against them
    return n_rays * len(times) / sum(times), times, threads


def eager_gpu_rates(sc, P, dev, steps=2, warmup=1, n_chunks=8):
    """The reference ALGORITHM (oracle port = the same eager torch ops the reference issues, F.grid_sample lookups, encoder
    hoisted) on this GPU: the stand-in for "the reference's PyTorch-GPU path" that the >=10x target names (/root/reference
    itself cannot travel to the GPU box).  fp32 with TF32 matmuls off and on (the authors' torch 1.11 defaulted to TF32)."""
    import torch
    from oracle import neo360_oracle as orc
    osc = orc.Scene(*[sc[k].to(dev) for k in ("planes_xz", "planes_xy", "planes_yz", "latent", "src_poses")],
                    float(sc["src_focal"][0]), float(sc["src_c"][0, 0]), float(sc["src_c"][0, 1]), IMG_W, IMG_H)
    Pd = {k: v.to(dev) for k, v in P.items()}
    o, d = frame_rays_cpu(0)
    n = n_chunks * CHUNK
    start = (IMG_H // 2) * IMG_W
    rays = {"rays_o": o[start:start + n].to(dev), "rays_d": d[start:start + n].to(dev), "viewdirs": d[start:start + n].to(dev)}
    res, outs = {"rays": n}, {}
    old = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32)
    for tf32 in (False, True):
        torch.backends.cuda.matmul.allow_tf32 = tf32
        torch.backends.cudnn.allow_tf32 = tf32
        with torch.no_grad():
            for _ in range(warmup):
                orc.render_chunked(rays, osc, Pd, N_COARSE, N_FINE, chunk=CHUNK, lookup_impl="aten")
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                out = orc.render_chunked(rays, osc, Pd, N_COARSE, N_FINE, chunk=CHUNK, lookup_impl="aten")
            e1.record()
            torch.cuda.synchronize()
        res["tf32" if tf32 else "fp32"] = n * steps / (e0.elapsed_time(e1) * 1e-3)
        outs[tf32] = out
    torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = old
    # the reference's own TF32-vs-fp32 deviation on these rays: the noise floor SURVEY.md 8(d) asks for
    res["tf32_vs_fp32_linf_rgb"] = float((outs[True]["comp_rgb"] - outs[False]["comp_rgb"]).abs().max())
    res["tf32_vs_fp32_psnr"] = orc.psnr(outs[True]["comp_rgb"].cpu(), outs[False]["comp_rgb"].cpu())
    res["note"] = "oracle port (reference algorithm, eager torch ops incl. F.grid_sample) on the same GPU, encoder hoisted, chunk=1024"
    del osc, Pd
    torch.cuda.empty_cache()
    return res


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    workload = "neo360 tri-planar render, 3 src views, 640x480, 128+64 samples (BASELINE configs[1])"

    if args.impl == "reference":
        if rank != 0:
            return
        sc, P = build_scene_cpu()
        rate, times, threads = cpu_reference_rate(sc, P, args.cpu_sample_rays, steps=args.steps, warmup=args.warmup)
        ms = 1e3 * sum(times) / len(times)
        line = {"impl": "reference", "metric": "rays/sec at 640x480, 192 samples/ray", "value": rate, "unit": "rays/s",
                "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": workload, "rays_per_step": args.cpu_sample_rays, "chunk": CHUNK,
                           "note": "reference algorithm = CPU oracle port (eager torch, F.grid_sample), encoder hoisted; each step a bounded sample of the frame"},
                "cpu_baseline": {"value": rate, "unit": "rays/s", "cores": threads, "kind": "port",
                                 "sample": f"{args.cpu_sample_rays} rays (one reference chunk) of frame 0 per step"},
                "e2e": {"value": rate, "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return

    if args.impl == "eager-gpu":
        if rank != 0:
            return
        import torch
        sc, P = build_scene_cpu()
        res = eager_gpu_rates(sc, P, torch.device("cuda", local), steps=args.steps, warmup=args.warmup)
        print(json.dumps({"impl": "eager-gpu", "metric": "rays/sec at 640x480, 192 samples/ray", "unit": "rays/s",
                          "value": res["fp32"], "value_tf32": res["tf32"], "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
                          "config": {"workload": workload, "rays_per_step": res["rays"], "chunk": CHUNK, "note": res["note"]},
                          "tf32_vs_fp32": {"linf_rgb": res["tf32_vs_fp32_linf_rgb"], "psnr": res["tf32_vs_fp32_psnr"]}}))
        return

    import torch
    import ctypes as C
    import numpy as np
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback for the product path)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    from neo360_b200 import NeRF_TP, _lib as L, build
    lib = L.load(build.build())

    if args.mode != "frames":
        import bench_modes
        line = bench_modes.run(args, rank, world, local, dev, dist, peaks())
        if rank == 0:
            print(json.dumps(line))
        if dist is not None:
            dist.destroy_process_group()
        return

    sc, P = build_scene_cpu()
    net = NeRF_TP(num_coarse_samples=N_COARSE, num_fine_samples=N_FINE, num_src_views=NV, precision=args.precision).eval()
    net.load_state_dict(P)
    net = net.to(dev)
    scene_keys = ("planes_xz", "planes_xy", "planes_yz", "latent", "src_poses", "src_focal", "src_c")
    torch.cuda.synchronize()
    t_prep = time.perf_counter()
    scene_dev = [sc[k].to(dev) for k in scene_keys]
    torch.cuda.synchronize()
    scene_h2d_ms = (time.perf_counter() - t_prep) * 1e3         # 0.56 GB of raw feature maps from pageable host memory
    prep = []
    for _ in range(3):                                          # first build is cold (module load, attribute setup); a scene change costs the warm figure
        torch.cuda.synchronize()
        t_prep = time.perf_counter()
        net.set_scene(*scene_dev, sc["img_wh"])
        torch.cuda.synchronize()
        prep.append((time.perf_counter() - t_prep) * 1e3)
    scene_prepare_cold_ms, scene_prepare_ms = prep[0], min(prep[1:])     # per scene, outside the timed region
    del scene_dev
    n = args.rays
    total_steps = args.warmup + args.steps
    # per-step inputs: a different turntable frame per (step, rank); pinned host copies for the e2e leg
    host = []
    for s in range(min(total_steps, 4)):
        o, d = frame_rays_cpu((s * world + rank) % 100)
        host.append((o[:n].contiguous().pin_memory(), d[:n].contiguous().pin_memory()))
    devrays = [{"rays_o": o.to(dev), "rays_d": d.to(dev), "viewdirs": d.to(dev)} for (o, d) in host]

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    wh = (IMG_W, IMG_H) if (n == IMG_W * IMG_H and not os.environ.get("NEO360_NO_BLOCK_ORDER")) else None

    last = {}

    def step_resident(s):
        last["out"] = net.render_rays_test(devrays[s % len(devrays)], chunk=CHUNK, img_wh=wh)

    in_o, in_d = torch.empty(n, 3, device=dev), torch.empty(n, 3, device=dev)        # device staging of the per-step inputs
    out_rgb, out_depth = torch.empty(n, 3).pin_memory(), torch.empty(n).pin_memory()   # contiguous pinned outputs (one DMA each)

    def step_e2e(s):
        o, d = host[s % len(host)]
        in_o.copy_(o, non_blocking=True)
        in_d.copy_(d, non_blocking=True)
        r = net.render_rays_test({"rays_o": in_o, "rays_d": in_d, "viewdirs": in_d}, chunk=CHUNK, img_wh=wh)
        out_rgb.copy_(r["rgb"], non_blocking=True)
        out_depth.copy_(r["depth"], non_blocking=True)
        return r

    def timed(fn, sampler=None):
        with torch.no_grad():
            for s in range(args.warmup):
                fn(s)
            barrier()
            if sampler:
                sampler.start()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for s in range(args.steps):
                fn(args.warmup + s)
            e1.record()
            barrier()
            if sampler:
                sampler.stop_flag = True
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if dist is not None:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    sampler = ClockSampler(local) if rank == 0 else None
    lib.neo_profile(0)
    ms_res = timed(step_resident, sampler)
    launches = C.c_ulonglong()
    lib.neo_profile_read(None, None, C.byref(launches), None)
    net.check()
    if args.dump_outputs and rank == 0:
        # 11 floats per ray: a whole frame is 13.5 MB, so every array is written in full
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, t in last["out"].items():
            np.save(os.path.join(args.dump_outputs, f"{name}.npy"), t.float().cpu().numpy())
    del last["out"]
    ms_e2e = timed(step_e2e)
    variants = {}
    if world == 1 and not args.no_extras and n == IMG_W * IMG_H:
        from neo360_b200 import ops
        pose_host = [__import__("neo360_b200").synth.target_pose(v, 100)[:3, :4].contiguous().pin_memory() for v in range(4)]

        def step_pose(s):
            # SURVEY.md 8(f3): rays generated on the device from the (3,4) pose (datasets/ray_utils.py:84-176) -- 48 bytes of H2D per frame
            c2w = pose_host[s % len(pose_host)].to(dev, non_blocking=True)
            ro, vd, rd, _ = ops.get_rays(IMG_H, IMG_W, 0.8 * IMG_W, c2w)
            r = net.render_rays_test({"rays_o": ro, "rays_d": rd, "viewdirs": vd}, chunk=CHUNK, img_wh=wh)
            out_rgb.copy_(r["rgb"], non_blocking=True)
            out_depth.copy_(r["depth"], non_blocking=True)

        def step_chunked(s):
            # the UNCHANGED reference render loop (models/neo360/model.py:861-896): one model(...) call per 1024-ray chunk
            o, d = host[s % len(host)]
            do, dd = o.to(dev, non_blocking=True), d.to(dev, non_blocking=True)
            outs = []
            for i in range(0, n, CHUNK):
                outs.append(net({"rays_o": do[i:i + CHUNK], "rays_d": dd[i:i + CHUNK], "viewdirs": dd[i:i + CHUNK]},
                                False, False, None, None, out_depth=True)[1])
            rgb = torch.cat([x[0] for x in outs]); dep = torch.cat([x[5] for x in outs])
            out_rgb.copy_(rgb, non_blocking=True)
            out_depth.copy_(dep, non_blocking=True)

        keep_steps, keep_warm = args.steps, args.warmup
        args.steps, args.warmup = 2, 1
        variants["pose_in_rays_on_device"] = {"value": n * args.steps / (timed(step_pose) * 1e-3), "unit": "rays/s", "h2d_bytes_per_step": 48,
                                              "note": "e2e with neo_get_rays on the device from an H2D (3,4) pose instead of host-built rays"}
        variants["per_chunk_calls"] = {"value": n * args.steps / (timed(step_chunked) * 1e-3), "unit": "rays/s", "calls_per_frame": (n + CHUNK - 1) // CHUNK,
                                       "note": "e2e through the reference's unchanged chunk loop: one NeRF_TP.forward per 1024 rays"}
        args.steps, args.warmup = keep_steps, keep_warm
    # roofline of the dominant kernel: CUDA events around every field launch, on the launching stream
    lib.neo_profile(1)
    with torch.no_grad():
        for s in range(args.steps):
            step_resident(args.warmup + s)
    fms, nf, _l, pts = C.c_float(), C.c_int(), C.c_ulonglong(), C.c_double()
    lib.neo_profile_read(C.byref(fms), C.byref(nf), C.byref(_l), C.byref(pts))
    lib.neo_profile(0)
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    pk = peaks()
    rays_total = n * args.steps * world
    value = rays_total / (ms_res * 1e-3)
    e2e = rays_total / (ms_e2e * 1e-3)
    # each field launch handles one branch; fg and bg launches alternate, so the mean flop/point is the fg/bg average
    flops_alg = pts.value * 0.5 * (FLOP_PER_POINT[0] + FLOP_PER_POINT[1])
    flops_issued = pts.value * 2.0 * ISSUED_MAC_PER_POINT if args.precision == "tc" else flops_alg
    ach = flops_issued / (fms.value * 1e-3) / 1e12                       # what the tensor pipe really does per second
    ach_ref = flops_alg / (fms.value * 1e-3) / 1e12                      # reference-formulation FLOPs per second of field-kernel time
    # reference-formulation figure with the per-scene pre-projection charged to ONE frame (SURVEY.md 8(d)'s condition for quoting it)
    ach_ref_charged = flops_alg / ((fms.value + args.steps * scene_prepare_ms) * 1e-3) / 1e12
    traffic = None
    tj = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tj):
        traffic = json.load(open(tj)).get(args.precision)
    line = {
        "metric": "rays/sec at 640x480, 192 samples/ray", "value": value, "unit": "rays/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_res / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None,
        "dtype": "f16 operands, f32 accumulate (tcgen05)" if args.precision == "tc" else "f32",
        "data": "synthetic",
        "config": {"workload": workload, "rays_per_step_per_gpu": n, "chunk": CHUNK, "precision": args.precision,
                   "parallelism": f"ray-sharded x{world} (one frame per rank, no collective)",
                   "l2": "inputs larger than L2 (feature maps + per-sample workspace >> 126 MB)",
                   "valid_headline": n == IMG_W * IMG_H},
        "roofline": {"bound": "tensor", "achieved": ach, "peak": pk["bf16_tflops"], "unit": "TFLOP/s",
                     "frac": ach / pk["bf16_tflops"], "traffic": traffic, "peak_source": pk["src"],
                     "kernel": "field kernel (lookups + MLP), %d launches, %.3f ms mean" % (nf.value, fms.value / max(nf.value, 1)),
                     "flops": "FLOPs the tensor pipe has to issue for the re-associated network (2*MAC: trunk on pre-projected maps, bilinear "
                              "blend, folded head; tile padding not counted) / CUDA-event time of the field launches",
                     "share_of_step": (fms.value / args.steps) / (ms_res / args.steps),
                     "effective_tflops": ach_ref, "effective_frac": ach_ref_charged / pk["bf16_tflops"],
                     "note": "effective_* = reference-formulation algorithmic FLOPs (2*MAC of NeRFPPMLP incl. the latent columns, SURVEY.md 8(d)); "
                             "effective_frac charges scene_prepare_ms (the warm per-scene pre-projection that removes those FLOPs; cold first build and H2D reported beside it) to every frame"},
        "scene_prepare_ms": scene_prepare_ms, "scene_prepare_cold_ms": scene_prepare_cold_ms, "scene_h2d_ms": scene_h2d_ms,
        "e2e": {"value": e2e, "unit": "rays/s", "h2d_bytes_per_step": 2 * n * 3 * 4, "d2h_bytes_per_step": n * 4 * 4,
                "ms_per_step": ms_e2e / args.steps},
        "gpu_launches": int(launches.value),
        "clocks": sampler.result(),
    }
    if not args.no_extras and world == 1:
        line["variants"] = variants
    if not args.no_cpu_baseline and world == 1:
        rate, times, threads = cpu_reference_rate(sc, P, args.cpu_sample_rays, steps=1, warmup=0)
        line["cpu_baseline"] = {"value": rate, "unit": "rays/s", "cores": threads, "kind": "port",
                                "sample": f"{args.cpu_sample_rays} rays (one reference chunk of frame 0), {times[0]:.1f} s"}
        # PSNR / L-inf of OUR pixels against the oracle's on exactly that sample (BASELINE.json: "... ; PSNR vs ref"):
        # the chunk is rendered the way the reference would (a standalone chunk of `chunk` rays, quirk Q1)
        from oracle import neo360_oracle as orc
        rays_cpu, ref = cpu_reference_rate.last
        with torch.no_grad():
            got = net.render_rays_test({k: v.to(dev) for k, v in rays_cpu.items()}, chunk=CHUNK)
        net.check()
        line["parity"] = {"rays": int(args.cpu_sample_rays), "vs": "oracle port (fp32, CPU) on the cpu_baseline sample",
                          "linf_rgb": float((got["rgb"].cpu() - ref["comp_rgb"]).abs().max()),
                          "linf_depth": float((got["depth"].cpu() - ref["depth"]).abs().max()),
                          "linf_acc": float((got["fg_acc"].cpu() - ref["fg_acc"]).abs().max()),
                          "psnr_vs_ref": orc.psnr(got["rgb"].cpu(), ref["comp_rgb"])}
    if not args.no_extras and world == 1:
        # the reference's eager-PyTorch formulation on this GPU: denominator of the >=10x target (SURVEY.md 8(d), BASELINE.md section 3)
        del net
        torch.cuda.empty_cache()
        eg = eager_gpu_rates(sc, P, dev)
        eg["speedup_vs_fp32"] = e2e / eg["fp32"]
        eg["speedup_vs_tf32"] = e2e / eg["tf32"]
        line["eager_gpu"] = eg
    print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
