#!/usr/bin/env python3
"""Headline benchmark of the path-tracing hot path on N B200s (one process per GPU).

    python bench.py --gpus 1 --steps K --warmup W [--config 2|cornell1080|1|3|4|5]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...      # the reference's own OpenCL-C kernels on the host cores

Default workload = BASELINE.json configs[1] (`--config 2`): Cornell box_Monkey, 1920x1080, 256 spp, maxBounce 4,
glossy monkey + glass wall + emitting lamp (the pinned material variant of SURVEY.md §8d), environment = the only
map in the reference checkout (600x300 preview; the 8k JPEG is missing upstream).  A "step" renders that whole
frame once.  Scene buffers are the committed fixtures produced by the reference's own FileManager/BVH.py
(tests/golden/make_golden.py); config 5 is generated (tests/synthetic.py) and its BVH built by the native builder.

value      Mrays/s, device time (CUDA events on the launching stream), inputs resident in HBM.
e2e        the same metric through the reference-facing call (KernelLauncher.launch_Raytracing) with HOST buffers:
           every step re-uploads scene + environment (caches invalidated), renders, and reads the image back.
roofline   dominant kernel = k_trace (one launch per wavefront iteration; timed on its own in one extra step rendered
           with a single sample stream, because the timed steps overlap two streams' kernels).  Configs 1-4 keep their scene in
           L1/L2/shared memory, so the bound is the SM ISSUE rate (SURVEY.md §8d): achieved = thread-instructions/s
           = (40 per box test + 80 per triangle test, counted by the production FAST traversal itself in a
           collect_stats pass) x rays of the k_trace launches / summed duration of those launches (CUDA events around
           every launch of one extra step); peak = SMs x 4 schedulers x 32 lanes x SM clock.  Config 5 (1.5 GB of
           nodes and triangles) is bound by HBM: achieved = bytes this layout must fetch per ray (32 B per node
           visit, 48 B per triangle test, 52 B of path state) / the same duration, against the measured copy peak.
           `traffic` = ncu-measured DRAM bytes of one mid-frame k_trace launch (profiles/roofline_traffic.json).
cpu_baseline  oracle/_ref (the reference's .cl compiled by g++) on the host cores, bounded sample.
parity_vs_single_gpu  (N > 1) the N-GPU image against the same frame rendered by rank 0 alone, at a reduced spp.
extra      the north-star target case (Cornell box, 1920x1080, 256 spp) timed the same way as `value`.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from tests import fixtures  # noqa: E402  (fixture loader only; no oracle import here)

CONFIGS = {
    "1": dict(scene="cornell", width=512, height=512, spp=16, max_bounce=4, ibl="preview",
              workload="BASELINE config 1: Cornell box 512x512 16spp maxBounce4"),
    "2": dict(scene="monkey_cfg2", width=1920, height=1080, spp=256, max_bounce=4, ibl="preview",
              workload="Cornell box_Monkey 1920x1080 256spp maxBounce4 (glossy monkey, glass wall, emissive lamp)"),
    "3": dict(scene="furnace_cfg3", width=1920, height=1080, spp=1024, max_bounce=4, ibl="grey",
              workload="BASELINE config 3: FurnaceHD under uniform IBL 1920x1080 1024spp maxBounce4"),
    "4": dict(scene="serre", width=3840, height=2160, spp=512, max_bounce=4, ibl="8k",
              workload="BASELINE config 4: Serre_leger 3840x2160 512spp maxBounce4, 8192x4096 environment stand-in"),
    "5": dict(scene="synthetic5m", width=3840, height=2160, spp=4096, max_bounce=4, ibl="preview",
              workload="BASELINE config 5: synthetic 5M-triangle height field 3840x2160 4096spp maxBounce4"),
    "cornell1080": dict(scene="cornell", width=1920, height=1080, spp=256, max_bounce=4, ibl="preview",
                        workload="north-star target: Cornell box 1920x1080 256spp maxBounce4"),
}
SEED = 0
SYNTH_PARAMS = dict(cam_x="0", cam_y="-7.5", cam_z="4.5", cam_rx="-32", cam_ry="0", cam_rz="0", cam_DOF="50",
                    sun_rx="60", sun_ry="0", sun_rz="30", sun_Power="0.8", IBL_Power="1.0")
INSTR_PER_BOX, INSTR_PER_TRI = 40.0, 80.0      # SURVEY.md §8d
NODE_BYTES, TRI_BYTES, STATE_BYTES = 32.0, 48.0, 52.0   # DESIGN.md §2: node record, triangle record, path state per ray


# --------------------------------------------------------------------------------------------------------
def load_workload(cfg):
    if cfg["scene"] == "synthetic5m":
        import ensem3a_openclraytracer_b200 as rt
        from tests.synthetic import height_field_scene
        sc = height_field_scene(1582, seed=0)
        sc["BVH"] = rt.build_bvh(sc["faceData"], sc["V_p"])
        sc["params"] = SYNTH_PARAMS
    else:
        sc = fixtures.load_scene(cfg["scene"])
    ibl = fixtures.load_ibl(cfg["ibl"])
    cam, env = fixtures.cam_env(sc["params"], cfg["width"], cfg["height"])
    return sc, ibl, cam, env


def public_config(cfg):
    """The workload, identically named by both arms."""
    return {k: cfg[k] for k in ("workload", "scene", "width", "height", "spp", "max_bounce", "ibl")}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def cpu_renderer():
    """(kind, render(sc, cam, env, img_dim, spp, max_bounce, ibl, i0, i1, nthreads) -> (image, rays)) of the CPU arm:
    oracle/_ref (the reference's own kernel text compiled by g++) when it is present, else the C restatement of
    oracle/ (bit-identical to it, tests/test_oracle_vs_ref.py).  The only place bench.py executes oracle/."""
    from oracle import ref_lib
    if ref_lib.available() and ref_lib.available("libclref_count.so"):
        def render(sc, cam, env, img_dim, spp, mb, ibl, i0, i1, nthreads, count=False):
            out, cnt = ref_lib.raytrace(sc, cam, env, img_dim, spp, mb, ibl, i0=i0, i1=i1, counters=count,
                                        nthreads=nthreads)
            return out, (cnt["rays"] if cnt else None)
        return "reference", render
    from oracle import oracle

    def render(sc, cam, env, img_dim, spp, mb, ibl, i0, i1, nthreads, count=False):
        out, cnt = oracle.render(sc, cam, env, img_dim, spp, mb, ibl, i0=i0, i1=i1, nthreads=nthreads)
        return out, cnt["rays"]
    return "port", render


def cpu_band(cfg):
    """Host-independent bounded sample of the workload: a band of rows through the middle of the frame, 16 spp."""
    W, H = cfg["width"], cfg["height"]
    rows = min(H, 96 if W * H <= 1920 * 1080 else 24)
    if cfg["scene"] == "synthetic5m":
        rows = 8
    i0 = (H // 2 - rows // 2) * W
    return rows, i0, i0 + rows * W


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.thread = [], None, None
        self.index = index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return
        self.thread = threading.Thread(target=self._pump, daemon=True)
        self.thread.start()

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0]))
                smax = float(f[1])
            except ValueError:
                continue
            for n, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons),
                "samples": len(sm)}


# --------------------------------------------------------------------------------------------------------
def run_reference_arm(args, cfg, rank):
    """--impl reference: the reference's own Kernels/*.cl (compiled by g++ into oracle/_ref) on every host core,
    on a bounded sample of the workload per step.  Executes oracle/ — allowed only here.  torchrun exports
    OMP_NUM_THREADS=1, so the thread count is passed explicitly."""
    if rank != 0:
        return
    kind, render = cpu_renderer()
    sc, ibl, cam, env = load_workload(cfg)
    W, H, mb = cfg["width"], cfg["height"], cfg["max_bounce"]
    cores = os.cpu_count() or 1
    spp = 16
    rows, i0, i1 = cpu_band(cfg)
    sample = f"{rows} rows x {W} px x {spp} spp of the workload frame (reference RNG), {cores} OpenMP threads"
    # ray count of the sample (untimed counting run; the kernel is deterministic)
    _, rays = render(sc, cam, env, W * H, spp, mb, ibl, i0, i1, cores, count=True)
    times = []
    for s in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        render(sc, cam, env, W * H, spp, mb, ibl, i0, i1, cores)
        dt = time.perf_counter() - t0
        if s >= args.warmup:
            times.append(dt)
    total = sum(times)
    mrays = rays * len(times) / total / 1e6
    line = {"impl": "reference", "metric": "Mrays/s", "value": mrays, "unit": "Mrays/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / len(times),
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": public_config(cfg), "reference_sample": sample,
            "samples_per_s": (i1 - i0) * spp * len(times) / total,
            "cpu_baseline": {"value": mrays, "unit": "Mrays/s", "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": mrays, "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


def cpu_baseline_leg(ctx, cfg, sc, ibl, cam, env):
    """Bounded CPU run of oracle/_ref beside the GPU number + parity of the same pixels."""
    import ensem3a_openclraytracer_b200 as rt
    kind, render = cpu_renderer()
    W, H, mb = cfg["width"], cfg["height"], cfg["max_bounce"]
    cores = os.cpu_count() or 1
    rows, i0, i1 = cpu_band(cfg)
    spp = 64 if W * H <= 1920 * 1080 else 16
    t0 = time.perf_counter()
    ref, _ = render(sc, cam, env, W * H, spp, mb, ibl, i0, i1, cores)
    dt = time.perf_counter() - t0
    # same pixels, same (reference) generator on the GPU: ray count + parity.  The reference's 20-entry stack drops
    # pushes on trees that need more (stack.cl:21-26): only the reference-order traversal reproduces that.
    deep = ctx.stats()["ref_stack_need"] > 20
    o = rt.make_opts(rng_mode=rt.RNG_REFERENCE, pixel_begin=i0, pixel_end=i1,
                     traversal=rt.TRAVERSAL_REFERENCE if deep else rt.TRAVERSAL_FAST)
    out = ctx.render(cam, env, W, H, spp, mb, opts=o)
    st = ctx.stats()
    a, b = out[3 * i0:3 * i1], ref[3 * i0:3 * i1]
    rel = np.abs(a - b) / np.maximum(np.abs(b), 1e-3)
    parity = {"pixels": i1 - i0, "spp": spp, "identical_frac": float(np.mean(a == b)), "max_rel": float(rel.max()),
              "rmse": float(np.sqrt(np.mean((a - b) ** 2))),
              "traversal": "reference order, 20-entry stack (tree needs more)" if deep else "fast"}
    base = {"value": st["rays"] / dt / 1e6, "unit": "Mrays/s", "cores": cores, "kind": kind,
            "sample": f"{rows} rows x {W} px x {spp} spp of the workload frame (reference RNG), {dt:.1f} s on {cores} "
                      f"OpenMP threads; samples/s {(i1 - i0) * spp / dt:.0f}"}
    return base, parity


# --------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200rt", choices=["b200rt", "reference"])
    ap.add_argument("--config", default="2", choices=sorted(CONFIGS), help="BASELINE config; 2 is the judged headline")
    ap.add_argument("--reduce", default="peer", choices=["nccl", "peer"], help="multi-GPU partial-sum reduction")
    ap.add_argument("--spp", type=int, default=0, help="debug only; overrides the config's spp")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the Cornell 1080p side measurement")
    ap.add_argument("--lean", action="store_true", help="long workloads (config 5): one end-to-end step, no warm-up step for it")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    cfg = dict(CONFIGS[args.config])
    if args.spp > 0:
        cfg["spp"] = args.spp

    if args.impl == "reference":
        run_reference_arm(args, cfg, rank)
        return

    import torch
    import torch.distributed as dist
    import ensem3a_openclraytracer_b200 as rt
    from ensem3a_openclraytracer_b200.multigpu import DistributedRenderer, split_range

    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    sc, ibl, cam, env = load_workload(cfg)
    W, H, spp, mb = cfg["width"], cfg["height"], cfg["spp"], cfg["max_bounce"]
    npix = W * H

    kl = rt.KernelLauncher(None, None, None, None, cuda_device=local)  # the reference-facing plugin object
    kl.rng_mode, kl.seed, kl.sample_streams = rt.RNG_PHILOX, SEED, -1
    kl.deep_trees = "nodrop"     # the measured configuration is the fast traversal on every tree (config 5 is deeper than
    #                              the reference's 20-entry stack; its default would switch to the reference-order walk)
    ctx = kl._ctx
    fixtures.upload(ctx, sc, ibl)
    scene_stats = ctx.stats()
    stream = torch.cuda.Stream(device=dev)   # every launch, event and collective below is issued on this stream
    torch.cuda.set_stream(stream)
    ctx.set_stream(stream.cuda_stream)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2
    out_dev = torch.zeros(npix * 3, dtype=torch.float32, device=dev)
    dr = DistributedRenderer(ctx, rank, world, reduce=args.reduce) if world > 1 else None
    philox = dict(rng_mode=rt.RNG_PHILOX, seed=SEED, sample_streams=-1)       # the timed configuration
    philox1 = dict(rng_mode=rt.RNG_PHILOX, seed=SEED, sample_streams=1)       # kernels timed / counted on their own

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def render_resident(cam_, env_, w_, h_, spp_):
        if dr is not None:
            return dr.render(cam_, env_, w_, h_, spp_, mb, **philox)
        ctx.render_device(cam_, env_, w_, h_, spp_, mb, out_dev.data_ptr(), rt.make_opts(**philox))
        return out_dev

    def timed(fn, steps, warmup):
        """(ms per step max over ranks, rays per step of the whole job, launches of this rank per step)"""
        for _ in range(warmup):
            fn()
        barrier()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        barrier()
        for a, b in ev:
            flush.fill_(1)                       # evict L2 between timed iterations (outside the event pair)
            a.record(stream)
            fn()
            b.record(stream)
        barrier()
        ms = sum(a.elapsed_time(b) for a, b in ev)
        st = ctx.stats()
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        # every rank traces the frame's primary rays (the cached primary hit); they count once for the job
        r = torch.tensor([float(st["rays"])], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dist.all_reduce(r, op=dist.ReduceOp.SUM)
        return float(t.item()) / steps, float(r.item()), st["kernel_launches"]

    # ---- box / triangle tests per ray of the production traversal (FAST), counted on the GPU over 2 spp -----------
    o = rt.make_opts(traversal=rt.TRAVERSAL_FAST, collect_stats=True, output=rt.OUT_SUMS, sample_begin=0,
                     sample_end=min(2, spp), **philox1)
    ctx.render_device(cam, env, W, H, spp, mb, out_dev.data_ptr(), o)
    st = ctx.stats()
    box_per_ray, tri_per_ray = st["box_tests"] / st["rays"], st["tri_tests"] / st["rays"]
    # the same rays in the reference's own walk (BVH.py's tree, right-first, no culling: MathLib.cl:234-288) — SURVEY 8d's
    # per-ray figure; the 5 M-triangle scene is skipped (seconds per sample in that order)
    ref_box_per_ray = ref_tri_per_ray = None
    if args.config != "5":
        o = rt.make_opts(traversal=rt.TRAVERSAL_REFERENCE, stack_cap=64, collect_stats=True, output=rt.OUT_SUMS, sample_begin=0,
                         sample_end=1, **philox1)
        ctx.render_device(cam, env, W, H, spp, mb, out_dev.data_ptr(), o)
        st = ctx.stats()
        ref_box_per_ray, ref_tri_per_ray = st["box_tests"] / st["rays"], st["tri_tests"] / st["rays"]

    # ---- device-resident timing ------------------------------------------------------------------------------
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ms_per_step, rays_all_ranks, launches_step = timed(lambda: render_resident(cam, env, W, H, spp), args.steps, args.warmup)
    clocks = sampler.stop() if rank == 0 else None
    streams_used = ctx.stats()["sample_streams"]
    rays_step = rays_all_ranks - (world - 1) * npix
    mrays = rays_step / ms_per_step / 1e3

    # ---- one profiled step: CUDA events around every k_shade / k_trace launch (roofline of the dominant kernel) -----
    if dr is None:
        ctx.render_device(cam, env, W, H, spp, mb, out_dev.data_ptr(), rt.make_opts(time_kernels=True, **philox1))
    else:
        s0, s1 = split_range(spp, world)[rank]
        ctx.render_device(cam, env, W, H, spp, mb, out_dev.data_ptr(),
                          rt.make_opts(time_kernels=True, output=rt.OUT_SUMS, sample_begin=s0, sample_end=s1, **philox1))
    barrier()
    stp = ctx.stats()

    # ---- N > 1: the N-GPU image against rank 0 rendering the same frame alone (reduced spp) ---------------------
    parity_multi = None
    if dr is not None:
        pspp = min(spp, 16)
        img = dr.render(cam, env, W, H, pspp, mb, **philox)
        barrier()
        if rank == 0:
            multi = img.cpu().numpy()
            ctx.render_device(cam, env, W, H, pspp, mb, out_dev.data_ptr(), rt.make_opts(**philox1))
            torch.cuda.synchronize()
            single = out_dev.cpu().numpy()
            rel = np.abs(multi - single) / np.maximum(np.abs(single), 1e-3)
            parity_multi = {"spp": pspp, "pixels": npix, "max_rel": float(rel.max()),
                            "rmse": float(np.sqrt(np.mean((multi - single) ** 2))),
                            "identical_frac": float(np.mean(multi == single)),
                            "note": "sample ranges are summed per GPU, then across GPUs: float addition order differs"}
        barrier()

    # ---- the north-star target case, timed like `value` ------------------------------------------------------------
    extra = None
    if not args.no_extra and args.config == "2":
        c2 = CONFIGS["cornell1080"]
        sc2, ibl2, cam2, env2 = load_workload(c2)
        fixtures.upload(ctx, sc2, ibl2)
        ctx.set_stream(stream.cuda_stream)
        ms2, rays2_all, _ = timed(lambda: render_resident(cam2, env2, c2["width"], c2["height"], c2["spp"]),
                                  max(2, min(args.steps, 5)), 2)
        rays2 = rays2_all - (world - 1) * c2["width"] * c2["height"]
        extra = {"cornell_1080p": {"workload": c2["workload"], "value": rays2 / ms2 / 1e3, "unit": "Mrays/s",
                                   "per_gpu": rays2 / ms2 / 1e3 / world, "ms_per_step": ms2, "n_gpus": world,
                                   "samples_per_s": c2["width"] * c2["height"] * c2["spp"] / (ms2 * 1e-3),
                                   "target": ">= 1000 Mrays/s per GPU (BASELINE.json north_star)"}}
        fixtures.upload(ctx, sc, ibl)
        ctx.set_stream(stream.cuda_stream)

    # ---- end to end through the plugin with host buffers ---------------------------------------------------------
    host_out = np.zeros(npix * 3, np.float32)
    pinned = torch.empty(npix * 3, dtype=torch.float32).pin_memory() if world > 1 else None
    h2d = sum(int(sc[k].nbytes) for k in ("V_p", "V_n", "V_uv", "faceData", "materialData", "BVH")) + int(ibl.nbytes) + 60
    d2h = npix * 3 * 4

    def step_e2e():
        ctx.invalidate()
        if dr is None:
            kl.launch_Raytracing(host_out, sc["V_p"], sc["V_n"], sc["V_uv"], sc["faceData"], sc["materialData"],
                                 sc["lightData"], sc["BVH"], cam, env, npix, spp, mb, ibl)
        else:
            fixtures.upload(ctx, sc, ibl)
            ctx.set_stream(stream.cuda_stream)
            img = dr.render(cam, env, W, H, spp, mb, **philox)
            if rank == 0:
                pinned.copy_(img, non_blocking=True)
            torch.cuda.synchronize()

    ctx.set_stream(None if dr is None else stream.cuda_stream)
    e2e_steps = 1 if args.lean else max(1, min(args.steps, 3))
    if not args.lean:
        step_e2e()
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        step_e2e()
    barrier()
    e2e_s = time.perf_counter() - t0
    te = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_mrays = rays_step * e2e_steps / float(te.item()) / 1e6

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel -----------------------------------------------------------------------------
    props = torch.cuda.get_device_properties(dev)
    sm_count = props.multi_processor_count
    sm_mhz = (clocks or {}).get("sm_max_mhz") or 1965.0
    n_trace = stp["wave_iterations"]                      # one k_trace launch per wavefront iteration
    trace_rays = stp["rays"] - npix                       # rank 0's rays minus the primary rays of k_primary
    trace_s = stp["trace_kernel_ms"] * 1e-3
    hbm_peak, hbm_src = measured_peak()
    traffic, ncu_view = None, None
    prof = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if os.path.exists(prof):
        try:
            pj = json.load(open(prof)).get("config_" + args.config, {})
            traffic = pj.get("k_trace_dram_bytes_per_launch")
            ncu_view = {k: v for k, v in pj.items() if k != "k_trace_dram_bytes_per_launch"} or None
        except Exception:
            traffic = None
    common = {"kernel": "k_trace", "launches_per_step": n_trace, "avg_launch_us": 1e3 * stp["trace_kernel_ms"] / max(n_trace, 1),
              "kernel_ms_per_step": stp["trace_kernel_ms"], "k_shade_ms_per_step": stp["shade_kernel_ms"],
              "k_primary_ms_per_step": stp["primary_ms"], "step_ms_profiled": stp["total_ms"],
              "share_of_step": stp["trace_kernel_ms"] / stp["total_ms"],
              "box_tests_per_ray": box_per_ray, "tri_tests_per_ray": tri_per_ray, "traffic": traffic, "ncu": ncu_view}
    bytes_per_ray = NODE_BYTES * box_per_ray / 2.0 + TRI_BYTES * tri_per_ray + STATE_BYTES
    if args.config == "5":
        achieved = trace_rays * bytes_per_ray / trace_s / 1e9
        roofline = {"bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak,
                    "peak_source": hbm_src, "bytes_per_ray": bytes_per_ray,
                    "note": "scene (1.5 GB) lives in HBM: bytes this layout fetches per ray = 32 B per node visit "
                            "(two box tests) + 48 B per triangle test + 52 B of path state"}
    else:
        instr_per_ray = INSTR_PER_BOX * box_per_ray + INSTR_PER_TRI * tri_per_ray
        achieved = trace_rays * instr_per_ray / trace_s / 1e9
        peak = sm_count * 4 * 32 * sm_mhz * 1e6 / 1e9
        roofline = {"bound": "issue", "achieved": achieved, "peak": peak, "unit": "Gthread-instr/s", "frac": achieved / peak,
                    "peak_source": f"{sm_count} SMs x 4 schedulers x 32 lanes x {sm_mhz:.0f} MHz",
                    "thread_instr_per_ray": instr_per_ray,
                    # the same work over the whole timed step (shading, compaction, reduce and all sample streams included)
                    "frac_of_whole_step": (rays_step - npix) / world * instr_per_ray / (ms_per_step * 1e-3) / 1e9 / peak,
                    "l2_bytes_per_ray_this_layout": bytes_per_ray,
                    "note": "scene is cache-resident (SURVEY 8d): the bound is the SM issue rate; algorithmic work = 40 "
                            "thread-instructions per box test + 80 per triangle test, counted on the production (FAST) "
                            "traversal of the production culling tree — work actually done, so frac falls when a better "
                            "tree removes work faster than it removes time (reference_work has SURVEY 8d's own figure)"}
        if ref_box_per_ray is not None:
            ref_instr = INSTR_PER_BOX * ref_box_per_ray + INSTR_PER_TRI * ref_tri_per_ray
            ref_achieved = trace_rays * ref_instr / trace_s / 1e9
            roofline["reference_work"] = {
                "box_tests_per_ray": ref_box_per_ray, "tri_tests_per_ray": ref_tri_per_ray, "thread_instr_per_ray": ref_instr,
                "achieved": ref_achieved, "frac": ref_achieved / peak,
                "note": "SURVEY 8d's per-ray figure: box / triangle tests the reference's own walk (right-first over BVH.py's "
                        "tree, no culling) spends on the same rays, counted on the GPU in reference order over 1 spp; "
                        "divided by the same k_trace time.  Work the task needs done, not work this kernel performs"}
    roofline.update(common)

    line = {
        "metric": "Mrays/s", "value": mrays, "unit": "Mrays/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": public_config(cfg),
        "impl_config": {"rng": "philox4x32-10 keyed (pixel,sample,bounce)",
                        "traversal": "fast: conservative walk of a SAH culling tree built over the caller's leaf boxes "
                                     "(csrc/cull_tree.cpp), exact Moeller-Trumbore on the leaves, winner validated with the "
                                     "reference's exact leaf-box test",
                        "pipeline": "k_primary, then (spp*(maxBounce+2)) x (k_shade, k_trace) wavefront iterations",
                        "partition": "sample ranges" if world > 1 else "single GPU",
                        "sample_streams": streams_used,
                        "reduce": args.reduce if world > 1 else None,
                        "l2": "256 MiB flush write between timed iterations", "scene_in_smem": bool(stp["scene_in_smem"]),
                        "triangles": scene_stats["triangles"], "bvh_depth": scene_stats["bvh_depth"],
                        "set_scene_repack_ms": scene_stats["repack_ms"]},
        "samples_per_s": npix * spp / (ms_per_step * 1e-3),
        "rays_per_step": rays_step, "rays_per_sample": rays_step / (npix * spp),
        "e2e": {"value": e2e_mrays, "unit": "Mrays/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": 1e3 * float(te.item()) / e2e_steps, "steps": e2e_steps},
        "gpu_launches": args.steps * (launches_step + (1 if world > 1 else 0)),
        "clocks": clocks, "roofline": roofline,
    }
    if parity_multi is not None:
        line["parity_vs_single_gpu"] = parity_multi
    if extra is not None:
        line["extra"] = extra
    if world == 1 and not args.no_cpu_baseline:
        ctx.set_stream(None)
        base, parity = cpu_baseline_leg(ctx, cfg, sc, ibl, cam, env)
        if base is not None:
            line["cpu_baseline"] = base
            line["parity_vs_reference"] = parity
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
