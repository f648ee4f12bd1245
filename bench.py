#!/usr/bin/env python
"""bench.py -- headline benchmark: path segments per second on the reference's sample scene.

Workload (BASELINE.json configs[1]): the shipped example scene (9 objects, diffuse + emissive), 800x800,
5000 samples per pixel, 8 bounces, stream compaction on.  One "step" = one whole render of that frame
(3.2e9 paths) on every rank.  With N ranks (torchrun, one per GPU) rank r renders samples [r*5000, (r+1)*5000)
of every pixel (sharding by sample index, weak scaling) and the per-GPU accumulation buffers are combined with
one NCCL reduce per step, inside the timed region.

  value         device-timed Mseg/s with everything resident in HBM (CUDA events on the launching stream)
  e2e           the same render through the public host API with HOST buffers: scene upload (H2D) + render +
                download of the float image (D2H) every step, wall clock around synchronised calls
  roofline      HBM roofline of the dominant kernels k_bounce / k_bounce_q (all launches of a step together), with the
                issue-slot roofline next to it (the kernels are issue-bound)
  strong        BASELINE configs[4]: 3840x2160, 16 384 spp IN TOTAL split by sample index over the N ranks, one NCCL
                reduce of the 133 MB float4 image inside the timed region (strong scaling; the headline is weak scaling)
  multi_gpu_check   (N > 1) before timing: a 200x200 frame rendered sharded + reduced equals the same samples on one GPU
  configs       (N = 1) BASELINE configs[2], [3] at 10 % of their sample counts, after the timed region
  shim_calls_per_s  (N = 1) the reference's own calling pattern: cudaRaytraceCore() once per sample at 800x800
  cpu_baseline  the CPU oracle (oracle/pt_oracle.c, "port") on a bounded sample of the same workload, rank 0, all host cores

`--impl reference` times the CPU implementation of the path on the host cores: the reference's own kernels are
TODO stubs (SURVEY.md 0), so this is the oracle port, which calls restatements of the reference's implemented
functions and our specification of the stubs.  It uses every core the process may run on (sched_getaffinity),
whatever OMP_NUM_THREADS says (torchrun sets it to 1).
"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "oracle")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

METRIC = "path segments per second, reference sample scene 800x800, 5000 spp, 8 bounces"
UNIT = "Mseg/s"
RES, SPP, DEPTH, SEED = 800, 5000, 8, 565
CPU_SPP = 32  # bounded CPU sample: 32 spp of the 800x800 frame (about 20 s of CPU work over the host cores)
WF_SPP = 50  # samples of the frame per wavefront: 32 M paths, 3.07 GB of path state (>> 126 MB L2); 100 wavefronts per step
STRONG_SCENE, STRONG_SPP, STRONG_WF_SPP = os.path.join("scenes", "sample_4k.txt"), 16384, 4
# BASELINE configs[2], [3]: (name, scene file or procedural:n, spp of the config, depth, samples per wavefront)
EXTRA_CONFIGS = [("cornell_glass_dof_1080p", os.path.join("scenes", "cornell_glass_dof.txt"), 4096, 12, 8),
                 ("procedural_10k_1080p", "procedural:10000", 1024, 8, 32),
                 # the headline scene once more, for its direct-light-sampling figure (`direct_light_sampling`)
                 ("sample_800", os.path.join("scenes", "sample.txt"), 5000, 8, 50)]
EXTRA_FRACTION = 0.1


def host_threads():
    """cores this process may run on -- NOT OMP_NUM_THREADS, which torchrun forces to 1"""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def load_sample_scene(pt):
    """The reference loader's parse of its own data/scenes/sampleScene.txt (tests/golden/ref_vectors.json)."""
    with open(os.path.join(ROOT, "tests", "golden", "ref_vectors.json")) as f:
        s = json.load(f)["scene"]
    g = np.frombuffer(bytes.fromhex(s["geoms_hex"]), dtype=pt.GEOM_DTYPE).copy()
    m = np.frombuffer(bytes.fromhex(s["materials_hex"]), dtype=pt.MATERIAL_DTYPE).copy()
    c = np.frombuffer(bytes.fromhex(s["camera_hex"]), dtype=pt.CAMERA_DTYPE).copy()
    return g, m, c


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def cpu_oracle_rate(threads=0, spp=CPU_SPP):
    """configs[0] scaled to a ~20 CPU-second sample: sample scene, 800x800, CPU_SPP spp, 8 bounces on the host
    cores through the oracle port; `threads` is passed to the OpenMP region explicitly."""
    from oracle_py import Oracle
    pt_dtypes = importlib.import_module("project3-pathtracer_b200")
    g, m, c = load_sample_scene(pt_dtypes)
    orc = Oracle()
    scn = orc.make_scene(g, m, c)
    nthreads = threads if threads > 0 else host_threads()
    _, live, secs = orc.render(scn, 0, spp, DEPTH, SEED, threads=nthreads)
    segs = int(live.sum())
    return segs, secs, nthreads


_JSON_FD = 1  # the process's original stdout (main() moves everything else to stderr)


def _emit(line):
    os.write(_JSON_FD, (line + "\n").encode())


def run_reference(args, rank):
    """--impl reference: the CPU path on the host cores (rank 0 only; the other ranks exit without work)."""
    if rank != 0:
        return
    rates, last = [], None
    for i in range(args.warmup + args.steps):
        segs, secs, nthreads = cpu_oracle_rate()
        if i >= args.warmup:
            rates.append((segs, secs))
        last = nthreads
    tot_s = sum(s for s, _ in rates)
    tot_t = sum(t for _, t in rates)
    val = tot_s / tot_t / 1e6
    sample = "sample scene 800x800, %d spp, 8 bounces per step (BASELINE configs[0] x %d); %d segments per step" % (CPU_SPP, CPU_SPP, rates[0][0])
    _emit(json.dumps({
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * tot_t / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "reference sample scene 800x800, 8 bounces; bounded sample: %d spp per step on host cores" % CPU_SPP,
                   "host_threads": last, "omp_num_threads_env_ignored": os.environ.get("OMP_NUM_THREADS")},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": last, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


def multi_gpu_check(pt, sh, torch, dist, geoms, mats, cam, rank, world, local, stream):
    """SURVEY 8e "Determinism": a 200x200 frame, 8*N spp sharded by sample index + one reduce, against the same samples on
    one GPU (rank 0): segment counts equal, images equal up to float summation order."""
    small = cam.copy()
    small["resolution"][0] = [200, 200]
    spp = 8 * world
    with pt.Context(geoms, mats, small, device=local) as c:
        sh.render_sharded(c, spp, DEPTH, SEED, rank, world, stream=stream)
        stream.synchronize()
        _, segs, _ = c.counters()
        t = torch.tensor([float(segs)], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        out = None
        if rank == 0:
            got = c.download_sum()
            c.clear()
            c.render(0, spp, DEPTH, SEED)
            want = c.download_sum()
            _, want_segs, _ = c.counters()
            rmse = float(np.sqrt(np.mean((got.astype(np.float64) - want) ** 2)))
            out = {"frame": "200x200", "spp_total": spp, "rmse": rmse, "max_sum": float(np.abs(want).max()),
                   "segments_sharded": int(t.item()), "segments_one_gpu": int(want_segs),
                   "segments_equal": int(t.item()) == int(want_segs),
                   "rmse_ok": rmse <= 1e-6 * max(1.0, float(np.abs(want).max()))}
        dist.barrier()
    if out is not None and not (out["segments_equal"] and out["rmse_ok"]):
        raise SystemExit("multi-GPU check failed: %s" % json.dumps(out))
    return out


def strong_leg(pt, sh, torch, dist, rank, world, local, stream, spp_total):
    """BASELINE configs[4]: 3840x2160, spp_total samples split by sample index over the ranks, one reduce, timed on the
    device from the first launch to the end of the reduce (max over ranks)."""
    sc = pt.Scene(os.path.join(ROOT, STRONG_SCENE))
    g, m, cam, _ = sc.frame(0)
    W, H = sc.width, sc.height
    ctx = pt.Context(g, m, cam, device=local)
    try:
        ctx.set_wavefront_paths(W * H * STRONG_WF_SPP)
        ctx.set_stream(stream.cuda_stream)
        accum = sh.accum_tensor(ctx)
        b, n = sh.sample_range(rank, world, spp_total)

        def combine():
            if world > 1:
                with torch.cuda.stream(stream):
                    sh.reduce_image(accum, dst=0)

        ctx.clear()
        ctx.render(b, min(n, 2 * STRONG_WF_SPP), DEPTH, SEED)  # warm-up: kernels, NCCL channel for this buffer
        combine()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ev0, evr, ev1 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        ctx.clear()
        ev0.record(stream)
        ctx.render(b, n, DEPTH, SEED)
        evr.record(stream)
        combine()
        ev1.record(stream)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ms, red = ev0.elapsed_time(ev1), evr.elapsed_time(ev1)
        paths, segs, _ = ctx.counters()
        t = torch.tensor([ms, red], device="cuda", dtype=torch.float64)
        tot = torch.tensor([float(segs), float(paths)], device="cuda", dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dist.all_reduce(tot, op=dist.ReduceOp.SUM)
        ms, red = (float(x) for x in t.tolist())
        segs_all, paths_all = (float(x) for x in tot.tolist())
        mean_lum = float(ctx.download_mean(spp_total).mean()) if rank == 0 else None
    finally:
        ctx.close()
    return {"workload": "%dx%d sample scene, %d spp in total, %d bounces (BASELINE configs[4])" % (W, H, spp_total, DEPTH),
            "scaling": "strong", "n_gpus": world, "spp_per_rank": n, "ms": ms, "Mseg_per_s": segs_all / ms / 1e3,
            "spp_per_s": spp_total / (ms * 1e-3), "segments": segs_all, "paths": paths_all,
            "reduce_ms": red, "reduce_bytes": W * H * 16 if world > 1 else 0,
            "reduce_note": "rank-local time from the end of its own render to the end of the reduce (includes waiting for the slowest rank), max over ranks",
            "mean_luminance": mean_lum}


def extra_configs(pt, peak):
    """BASELINE configs[2], [3] (and the headline scene) at EXTRA_FRACTION of their sample counts (one GPU, device-timed),
    each without and with direct light sampling."""
    out = []
    for name, path, spp_full, depth, wf_spp in EXTRA_CONFIGS:
        try:
            if path.startswith("procedural:"):
                n = int(path.split(":")[1])
                tmp = os.path.join(tempfile.gettempdir(), "procedural_%d.txt" % n)
                subprocess.check_call([sys.executable, os.path.join(ROOT, "scenes", "gen_scenes.py"), "--procedural", str(n), tmp],
                                      stdout=subprocess.DEVNULL)
                path = tmp
            else:
                path = os.path.join(ROOT, path)
            sc = pt.Scene(path)
            g, m, cam, lens = sc.frame(0)
            spp = max(1, int(round(spp_full * EXTRA_FRACTION)))
            t0 = time.perf_counter()
            with pt.Context(g, m, cam, lens=lens if lens[0] > 0 else None) as ctx:
                t_ctx = time.perf_counter() - t0
                ctx.set_wavefront_paths(sc.width * sc.height * wf_spp)
                ctx.render(0, min(spp, wf_spp), depth, SEED)  # warm-up
                ctx.sync()
                ctx.clear()
                ctx.render(0, spp, depth, SEED)
                ms = ctx.last_render_ms()
                paths, segs, _ = ctx.counters()
                fb = ctx.filter_stats()
                retries = ctx.filter_retries()
                # the same frame with direct light sampling (DESIGN.md 4): shadow rays are traced from a queue by
                # launches of their own and counted apart from path segments
                direct = None
                try:
                    ctx.set_direct_lighting(True)
                    ctx.clear()
                    ctx.render(0, min(spp, wf_spp), depth, SEED)  # warm-up (allocates the shadow queues)
                    ctx.sync()
                    ctx.clear()
                    ctx.render(0, spp, depth, SEED)
                    ms_d = ctx.last_render_ms()
                    _, segs_d, _ = ctx.counters()
                    shadow, n_lights = ctx.shadow_rays()
                    direct = {"Mseg_per_s": segs_d / ms_d / 1e3, "Mrays_per_s": (segs_d + shadow) / ms_d / 1e3,
                              "shadow_rays": int(shadow), "lights": int(n_lights), "ms": ms_d,
                              "cost_vs_paths_only": (ms_d / max(1, segs_d)) / (ms / max(1, segs))}
                except Exception as e:
                    direct = {"error": str(e)}
            alg = 96.0 * (segs - paths) + 32.0 * paths
            line = {"name": name, "geoms": int(sc.n_geoms), "resolution": [sc.width, sc.height], "spp": spp,
                    "spp_of_config": spp_full, "depth": depth, "ms": ms, "Mseg_per_s": segs / ms / 1e3,
                    "spp_per_s": spp / (ms * 1e-3), "segments": int(segs), "fallback_fraction": fb / max(1, segs),
                    "retry_fraction": retries / max(1, segs), "roofline_frac": alg / (ms * 1e-3) / 1e9 / peak, "context_create_s": t_ctx}
            line["direct_light_sampling"] = direct
            if sc.n_geoms > 32:
                line["bound"] = "latency / FP32 (hierarchy traversal): the HBM fraction is reported for completeness only"
            out.append(line)
        except Exception as e:  # a side measurement never takes the headline down
            out.append({"name": name, "error": str(e)})
    return out


def shim_rate(pt, geoms, mats, cam, calls=1000, warm=32):
    """the reference's calling pattern (src/main.cpp:93-113): cudaRaytraceCore() once per sample, host image updated
    with the running mean on every call.  Steady state of one long sequence: the first `warm` iterations (context
    creation, the first groups of samples traced ahead) are not timed."""
    compat = importlib.import_module("project3-pathtracer_b200.compat")
    rs = compat.RefScene([(geoms, cam)], mats, iterations=SPP)  # ITERATIONS 5000, as the scene file says
    compat.reset(); compat.set_trace_depth(DEPTH); compat.set_seed(SEED); compat.set_exit_on_error(False)
    try:
        for k in range(1, warm + 1):
            compat.cudaRaytraceCore(None, rs.camera, 0, k, rs.materials, len(rs.materials), rs.geoms, len(rs.geoms))
        t0 = time.perf_counter()
        for k in range(warm + 1, warm + calls + 1):
            compat.cudaRaytraceCore(None, rs.camera, 0, k, rs.materials, len(rs.materials), rs.geoms, len(rs.geoms))
        dt = time.perf_counter() - t0
        if compat.last_status() != 0:
            raise RuntimeError("cudaRaytraceCore status %d" % compat.last_status())
        return {"calls": calls, "calls_per_s": calls / dt, "ms_per_call": 1e3 * dt / calls,
                "mean_of_running_mean": float(rs.image.mean()),
                "note": "800x800, iterations %d..%d of one sequence, %d bounces, D2H of the 7.68 MB running mean every call; "
                        "samples traced ahead in groups of 8 (pt_stream_*)" % (warm + 1, warm + calls, DEPTH)}
    finally:
        compat.reset()


def dump_outputs(out_dir, ctx, live):
    """What a caller of the timed path receives after its last step (rank 0; with N ranks the image is the reduced one):
    the summed radiance image (download_sum, 800*800 x 3 float32, 7.7 MB) and the live paths per depth (counters)."""
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "image_sum.npy"), ctx.download_sum())
    np.save(os.path.join(out_dir, "live_per_depth.npy"), live[:DEPTH].astype(np.float64))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--spp", type=int, default=SPP)
    ap.add_argument("--wf-spp", type=int, default=WF_SPP)
    ap.add_argument("--strong-spp", type=int, default=STRONG_SPP, help="total samples of the 4K strong-scaling leg (0 = skip)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the strong leg, the other configs and the shim rate")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed to DIR/<name>.npy (the inputs are fixed and seeded, so "
                         "two builds can be compared output for output)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    # stdout carries exactly ONE line, the JSON: libraries that write to file descriptor 1 on their own (NCCL prints
    # "NCCL version ..." there when NCCL_DEBUG is set) are sent to stderr instead
    global _JSON_FD
    sys.stdout.flush()
    _JSON_FD = os.dup(1)
    os.dup2(2, 1)
    if args.impl == "reference":
        run_reference(args, rank)
        return

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the path tracer has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    pt = importlib.import_module("project3-pathtracer_b200")
    geoms, mats, cam = load_sample_scene(pt)
    npix = RES * RES
    ctx = pt.Context(geoms, mats, cam, device=local)
    ctx.set_wavefront_paths(npix * args.wf_spp)
    stream = torch.cuda.Stream()
    ctx.set_stream(stream.cuda_stream)
    sh = importlib.import_module("project3-pathtracer_b200.sharding")
    accum = sh.accum_tensor(ctx)  # zero-copy view of the float4 accumulation image in HBM
    first_sample = rank * args.spp

    mg_check = None
    if world > 1:
        mg_check = multi_gpu_check(pt, sh, torch, dist, geoms, mats, cam, rank, world, local, stream)

    def step():
        ctx.clear()
        ctx.render(first_sample, args.spp, DEPTH, SEED)
        if world > 1:
            with torch.cuda.stream(stream):
                sh.reduce_image(accum, dst=0)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-timed: K whole renders, scene and buffers resident ----
    for _ in range(args.warmup):
        step()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches0 = ctx.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    for _ in range(args.steps):
        step()
    ev1.record(stream)
    barrier()
    ms = ev0.elapsed_time(ev1)
    launches = ctx.launch_count() - launches0
    clocks = sampler.stop() if rank == 0 else None
    paths, segs, live = ctx.counters()  # of the last step (clear() resets them)
    t = torch.tensor([ms], device="cuda", dtype=torch.float64)
    tot = torch.tensor([float(segs), float(paths), float(launches)], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    ms = float(t.item())
    segs_all, paths_all, launches_all = (float(x) for x in tot.tolist())
    ms_per_step = ms / args.steps
    value = segs_all / (ms_per_step * 1e-3) / 1e6
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, ctx, live)

    # ---- end to end through the host API: H2D scene + render + D2H image, every step ----
    host_img = torch.empty((npix, 3), dtype=torch.float32).pin_memory()
    host_np = host_img.numpy()
    hg = torch.from_numpy(geoms.view(np.uint8)).pin_memory().numpy().view(pt.GEOM_DTYPE)
    hm = torch.from_numpy(mats.view(np.uint8)).pin_memory().numpy().view(pt.MATERIAL_DTYPE)
    hc = torch.from_numpy(cam.view(np.uint8)).pin_memory().numpy().view(pt.CAMERA_DTYPE)
    h2d = int(hg.nbytes + hm.nbytes + hc.nbytes)
    d2h = int(host_np.nbytes)

    def e2e_step():
        ctx.update_scene(hg, hm, hc)
        step()
        ctx.download_mean(args.spp * world if rank == 0 else args.spp, out=host_np)

    e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        e2e_step()
    barrier()
    e2e_s = time.perf_counter() - t0
    te = torch.tensor([e2e_s], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_s = float(te.item())
    e2e_value = segs_all * args.steps / e2e_s / 1e6
    ctx.close()

    # ---- strong scaling: the 4K frame, a fixed total of samples split over the ranks ----
    strong = None
    if not args.no_extras and args.strong_spp > 0:
        try:
            strong = strong_leg(pt, sh, torch, dist, rank, world, local, stream, args.strong_spp)
        except Exception as e:
            strong = {"error": str(e)}
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()  # rank 0 goes on to the host-side measurements; the other ranks are done

    if rank == 0:
        # roofline of the bounce kernels: algorithmic path-state bytes (SURVEY.md 8d) over all their launches of one step
        P1, S1 = float(paths), float(segs)
        alg_bytes = 96.0 * (S1 - P1) + 32.0 * P1
        peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(peaks_path):
            peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        else:
            peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
        achieved = alg_bytes / (ms_per_step * 1e-3) / 1e9
        n_bounce = max(1, (launches // args.steps) * DEPTH // (DEPTH + 1))  # launches per step = wavefronts * (DEPTH bounce kernels + 1 k_accum_counts)
        traffic, traffic_note, pipes, issue = None, "no ncu capture on file", None, None
        tpath = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tpath):
            tj = json.load(open(tpath))
            # DRAM bytes of one average bounce launch = measured DRAM/algorithmic ratio of the captured launch x the
            # algorithmic bytes of an average launch of this run
            traffic = tj["dram_over_algorithmic"] * alg_bytes / n_bounce
            traffic_note = "ncu dram read+write / algorithmic = %.3f on the captured launch (%s)" % (tj["dram_over_algorithmic"], tj["source"])
            pipes = tj.get("pipes_pct_of_peak")  # SURVEY 8d: FP32 pipe utilisation next to the HBM fraction (same capture)
            wps = tj.get("warp_inst_per_segment")  # all launches of one wavefront / its segments (ncu, deterministic)
            if wps and clocks and clocks.get("sm_mhz"):
                sm_count = tj.get("sm_count", 148)
                inst_per_s = wps * S1 / (ms_per_step * 1e-3)
                slots_per_s = sm_count * 4 * clocks["sm_mhz"] * 1e6
                issue = {"bound": "issue slots", "achieved": inst_per_s / 1e9, "peak": slots_per_s / 1e9, "unit": "G warp-inst/s",
                         "frac": inst_per_s / slots_per_s, "warp_inst_per_segment": wps,
                         "note": "warp instructions per segment from the ncu launch list of one wavefront (%s) x segments/s of this run; "
                                 "peak = %d SMs x 4 schedulers x the SM clock sampled during the timed region" % (tj.get("inst_source", tj["source"]), sm_count)}
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "reference sample scene (9 objects) %dx%d, %d spp per GPU, %d bounces, compaction on"
                                   % (RES, RES, args.spp, DEPTH),
                       "sharding": "by sample index; one NCCL reduce of the float4 image per step" if world > 1 else "single GPU",
                       "wavefront_paths": npix * args.wf_spp,
                       "l2": "path state per wavefront %.0f MB > 126 MB L2 (no flush needed)" % (npix * args.wf_spp * 96 / 1e6),
                       "seed": SEED},
            "spp_per_s": args.spp * world / (ms_per_step * 1e-3),
            "segments_per_step": segs_all, "paths_per_step": paths_all,
            "live_per_depth": [int(x) for x in live[:DEPTH]],
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "gpu_launches": int(launches_all),
            "clocks": clocks,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "frac_of_nominal_8000": achieved / 8000.0,
                         "traffic": traffic, "traffic_note": traffic_note, "peak_source": peak_src,
                         "kernel": "k_bounce (depth 0) + k_bounce_q (depths >= 1)",
                         "ncu_pipes_pct_of_peak": pipes,
                         "algorithmic_bytes_per_launch": alg_bytes / n_bounce, "launches_per_step": n_bounce,
                         "avg_launch_us": 1e3 * ms_per_step / n_bounce,
                         "note": "achieved = algorithmic bytes 96*(S-P) + 32*P of a step / CUDA-event time of the step; the step is "
                                 "%d bounce-kernel launches (99.9 %% of its GPU time), two wavefronts in "
                                 "flight on two streams, so this is bytes per average launch / (step time / launches)" % n_bounce},
            "issue_roofline": issue,
            "strong": strong,
        }
        if mg_check is not None:
            out["multi_gpu_check"] = mg_check
        if world == 1 and not args.no_extras:
            out["configs"] = extra_configs(pt, peak)
            try:
                out["shim_calls_per_s"] = shim_rate(pt, geoms, mats, cam)
            except Exception as e:
                out["shim_calls_per_s"] = {"error": str(e)}
        if not args.no_cpu_baseline:
            csegs, csecs, cthreads = cpu_oracle_rate()
            out["cpu_baseline"] = {"value": csegs / csecs / 1e6, "unit": UNIT, "cores": cthreads, "kind": "port",
                                   "sample": "BASELINE configs[0] x %d: sample scene 800x800, %d spp, 8 bounces (%d segments, %.2f s)"
                                             % (CPU_SPP, CPU_SPP, csegs, csecs)}
            if world == 1:
                s1, t1, _ = cpu_oracle_rate(threads=1, spp=2)  # SURVEY 8d: the same oracle on ONE core
                out["cpu_baseline_1core"] = {"value": s1 / t1 / 1e6, "unit": UNIT, "cores": 1, "kind": "port",
                                             "sample": "sample scene 800x800, 2 spp, 8 bounces (%d segments, %.2f s)" % (s1, t1)}
        if world == 1 and not args.no_cpu_baseline and not args.no_extras:
            # the other kernel the north star asks a roofline for: the stable stream-compaction primitive (an HBM-bound
            # kernel by nature), device-timed on its own, outside the timed region above
            try:
                n_c, keep = 1 << 27, 0.7
                rng = np.random.default_rng(1)
                vals = rng.integers(0, 2 ** 32, n_c, dtype=np.uint32)
                flg = (rng.random(n_c, dtype=np.float32) < keep).astype(np.uint8)
                kept, cms = pt.compact_u32_timed(vals, flg, iters=10)
                cbytes = 5.0 * n_c + 4.0 * len(kept)
                out["compaction_primitive"] = {
                    "kernels": "k_compact_count + k_compact_scan + k_compact_scatter (pt_compact_u32)", "elements": n_c,
                    "keep": keep, "ms": cms, "Gelem_per_s": n_c / cms / 1e6, "bound": "hbm", "achieved": cbytes / cms / 1e6,
                    "peak": peak, "unit": "GB/s", "frac": cbytes / cms / 1e6 / peak,
                    "algorithmic_bytes": "5 B read per element + 4 B written per kept element"}
                del vals, flg, kept
            except Exception as e:  # never let the side measurement take the headline line down
                out["compaction_primitive"] = {"error": str(e)}
        _emit(json.dumps(out))


if __name__ == "__main__":
    main()
