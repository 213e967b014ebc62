#!/usr/bin/env python
"""Headline benchmark of the B200 path_tracer hot path (BASELINE.json metric: Msamples/s).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--spp-per-step S] [--dump-outputs DIR]

Workload (config C1 of BASELINE.json): Cornell box + 868,480-triangle Lambert mesh (procedural stand-in for the
Stanford dragon, see tungsten_b200/synth.py), 1920x1080, path_tracer, max_bounces 64, Sobol sampler,
target 1024 spp.  One STEP = one pass of the hot path over one batch: 64 samples per pixel of the whole frame
(132.7 M camera paths); the default 16 timed steps are the complete 1024-spp frame.  With N GPUs the image's
16x16 tiles are dealt round-robin to the ranks and a step renders 64*N spp (fixed work per GPU: weak scaling),
followed by the path's single collective, an all-gather of the tile-major float3 framebuffer.

`value`   : whole-job Msamples/s with everything resident in HBM (framebuffer stays on the device).
`e2e`     : the same metric through the reference-facing C-ABI call tgb200_render_tiles with HOST buffers
            (running-mean framebuffer + counts copied host->device and back inside every step).
`roofline`: traversal kernel (k_trace): algorithmic bytes = 48 B per closest-hit query (32 B ray read + 16 B hit
            write, SURVEY 8d) / CUDA-event duration of the launches in the timed region / measured HBM peak.
`cpu_baseline`: the reference's own CPU renderer (oracle/_ref/tungsten, built from /root/reference by
            oracle/ref/Makefile) on this box's host cores, same scene, bounded sample (fewer spp).
`--dump-outputs DIR`: after the timed steps, the framebuffer a caller reads back from the last one (running mean and
            sample count of every pixel, the whole frame gathered on rank 0) as DIR/mean.npy and DIR/count.npy (float32).
            Scene and seed are fixed, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import re
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

W, H = 1920, 1080
ALG_BYTES_PER_QUERY = 48
DUMP_LIMIT_BYTES = 64 << 20         # --dump-outputs: larger frames are written as a fixed, seeded sample of pixels
DUMP_SAMPLE_PIXELS = 1 << 21
CONFIGS = {
    "c1": {"res": (1920, 1080), "label": "C1: Cornell box + 868,480-tri Lambert mesh (procedural dragon stand-in), 1920x1080, path_tracer, max_bounces 64, Sobol"},
    "c2": {"res": (1920, 1080), "label": "C2: room with 327,680-triangle furniture stand-ins in rough conductor / rough dielectric / plastic / rough plastic, checker floor, quad + mesh lights + importance-sampled HDR environment, 1920x1080, max_bounces 16, Sobol"},
    "c3": {"res": (3840, 2160), "label": "C3: 12,544,000-triangle instanced forest (490 trees x 2 masters, flattened), Lambert + rough plastic + HDR sky, 3840x2160, max_bounces 16, Sobol"},
    "c4": {"res": (1920, 1080), "label": "C4: 650,000 quadratic B-spline curve segments (10,000 curly strands x 67 nodes, bcsdf_cylinder) with the hair BCSDF over a Lambert floor, quad light + constant sky, 1920x1080, max_bounces 16, Sobol"},
}


def _clock_sampler(stop, out, idx):
    q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
    while not stop.is_set():
        try:
            r = subprocess.run(["nvidia-smi", "-i", str(idx), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                               stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=5)
            f = [x.strip() for x in r.stdout.strip().split(",")]
            if len(f) >= 6:
                out.append(f)
        except Exception:
            pass
        stop.wait(0.2)


def _summarise_clocks(samples):
    if not samples:
        return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
    sm = sorted(int(s[0]) for s in samples if s[0].isdigit())
    names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
    reasons = [n for i, n in enumerate(names) if any(s[2 + i].lower().startswith("active") for s in samples)]
    return {"sm_mhz": sm[len(sm)//2] if sm else None, "sm_max_mhz": int(samples[0][1]) if samples[0][1].isdigit() else None,
            "reasons": reasons, "samples": len(samples)}


def _scene_dir():
    d = os.path.join(tempfile.gettempdir(), "tgb200_bench_scene")
    os.makedirs(d, exist_ok=True)
    return d


def make_scene(spp, config="c1"):
    from tungsten_b200 import synth
    d = _scene_dir()
    if config == "c3":
        path = os.path.join(d, "forest10m.json")
        if not os.path.exists(path):
            synth.instanced_forest(d, "forest10m", n_instances=490, tree_subdiv=5, res=CONFIGS["c3"]["res"], spp=spp, extent=40.0)
        return path
    if config == "c2":
        path = os.path.join(d, "room.json")
        if not os.path.exists(path):
            synth.save_rgbe(os.path.join(d, "room_env.hdr"), synth.sky_envmap(512, 256))
            synth.material_room(d, "room", res=CONFIGS["c2"]["res"], spp=spp, max_bounces=16, subdiv=6, env="room_env.hdr")
        return path
    if config == "c4":
        path = os.path.join(d, "hair650k.json")
        if not os.path.exists(path):
            synth.hair_scene(d, "hair650k", n_curves=10000, nodes_per_curve=67, res=CONFIGS["c4"]["res"], spp=spp, width=0.004)
        return path
    path = os.path.join(d, "cornell_dragon.json")
    marker = os.path.join(d, "cornell_dragon_body.wo3")
    if not (os.path.exists(path) and os.path.exists(marker)):
        synth.cornell_dragon_standin(d, res=(W, H), spp=spp)
    return path


def hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def parse_duration(text):
    """Seconds from the reference's `durationToString` (src/core/io/StringUtils.cpp:51-68):
    "[Dd ][Hh ][Mm ]Ss MSms" when >= 1 s, else the plain double followed by "s"."""
    m = re.search(r"Render time ((?:\d+d )?(?:\d+h )?(?:\d+m )?)(\d+)s (\d+)ms", text)
    if m:
        secs = float(m.group(2)) + float(m.group(3))/1e3
        for tok in m.group(1).split():
            secs += float(tok[:-1])*{"d": 86400.0, "h": 3600.0, "m": 60.0}[tok[-1]]
        return secs
    m = re.search(r"Render time ([0-9.eE+-]+)s", text)
    return float(m.group(1)) if m else None


def host_cpu_info():
    """What the CPU arm can actually use: affinity mask, cgroup quota, model string."""
    info = {"os_cpu_count": os.cpu_count() or 1}
    try:
        info["affinity"] = len(os.sched_getaffinity(0))
    except Exception:
        info["affinity"] = info["os_cpu_count"]
    quota = None
    for p in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(p).read().split()
            if p.endswith("cpu.max"):
                if txt[0] != "max":
                    quota = float(txt[0])/float(txt[1])
            else:
                q = float(txt[0])
                if q > 0:
                    quota = q/float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            break
        except Exception:
            continue
    info["cgroup_cpus"] = quota
    try:
        for ln in open("/proc/cpuinfo"):
            if ln.startswith("model name"):
                info["model"] = ln.split(":", 1)[1].strip(); break
    except Exception:
        pass
    usable = info["affinity"]
    if quota:
        usable = max(1, min(usable, int(quota + 0.5)))
    info["usable"] = usable
    return info


def run_reference_binary(scene_path, spp, threads):
    """Times oracle/_ref/tungsten (the unmodified reference) on `spp` samples per pixel of the bench scene.
    Returns (Msamples/s, render seconds): the reference's own "Render time", which excludes scene load and its
    Embree BVH build (src/tungsten/Shared.hpp:255-319) -- as our arm's timed region excludes tgb200_create."""
    exe = os.path.join(ROOT, "oracle", "_ref", "tungsten")
    if not os.path.exists(exe):
        return None
    js = json.load(open(scene_path))
    js["renderer"].update(spp=spp, spp_step=spp, adaptive_sampling=False, stratified_sampler=True,
                          hdr_output_file="ref.pfm", output_file="ref.png")
    d = os.path.dirname(scene_path)
    rp = os.path.join(d, "ref_run.json")
    json.dump(js, open(rp, "w"))
    out = subprocess.run([exe, "-t", str(threads), "-d", os.path.join(d, "ref_out"), rp], stdout=subprocess.PIPE,
                         stderr=subprocess.STDOUT, text=True)
    secs = parse_duration(out.stdout)
    if not secs:
        return None
    return W*H*spp/secs/1e6, secs


def bench_reference(args, rank, world):
    """--impl reference: the reference's own CPU path on the host cores (rank 0 only).  One step = one run of the
    unmodified binary on a bounded sample (spp chosen from a calibration run so that a step RENDERS for >= ~6 s)."""
    if rank != 0:
        return
    cpu = host_cpu_info()
    threads = cpu["usable"]
    scene_path = make_scene(1024, args.config)
    cal = run_reference_binary(scene_path, 2, threads)          # calibration, untimed
    if cal is None:
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/tungsten is missing (run make -C oracle/ref)"}))
        return
    spp = args.ref_spp if args.ref_spp > 0 else int(min(256, max(4, round(cal[0]*1e6*args.ref_seconds/(W*H)))))
    runs = []
    for i in range(args.warmup + args.steps):
        r = run_reference_binary(scene_path, spp if i >= args.warmup else 1, threads)
        if r is None:
            print(json.dumps({"impl": "reference", "unavailable": "the reference binary printed no render time"}))
            return
        if i >= args.warmup:
            runs.append(r)
    secs = sum(v[1] for v in runs)
    value = W*H*spp*len(runs)/secs/1e6
    rates = sorted(v[0] for v in runs)
    line = {"impl": "reference", "metric": "Msamples/sec (paths x spp)", "value": value, "unit": "Msamples/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3*secs/len(runs),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": CONFIGS[args.config]["label"]},
            "cpu_baseline": {"value": value, "unit": "Msamples/s", "cores": threads, "kind": "reference",
                             "sample": "%d spp of the whole %dx%d frame per step (bounded sample of the job; non-adaptive, so the per-sample rate is "
                                       "spp independent), tungsten -t %d, SSE4.2 Embree build without AVX (the reference's own ISA policy); time = the "
                                       "binary's 'Render time' (excludes scene load + BVH build, as our arm excludes tgb200_create)" % (spp, W, H, threads),
                             "min": rates[0], "median": rates[len(rates)//2], "max": rates[-1], "runs": len(rates),
                             "host": cpu},
            "e2e": {"value": value, "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


# ---- algorithmic bytes per unit of the non-traversal kernels (DESIGN.md section 5; 16-byte records T0..T3, E, pcg) -------------
STREAM_BYTES = {
    # new camera path: T0..T3 (64) + E (16) + pcg (8) + order (4) written
    "k_regen": {"bytes_per_unit": 92, "unit": "camera path started"},
    # path-bounce: T0..T3 + pcg read (72), T0/T1/T3 + pcg written (56), NEE/MIS scratch P,N0,N1,M0,M1,D0,D1 + vis written (120)
    "k_shade": {"bytes_per_unit": 248, "unit": "path ray shaded"},
    # path-bounce: T1,T3,E read (48) + vis,N1,M1,D0,D1 (72) ; survivor: T0 + pcg read (24), T0..T3,E,pcg,key written (92)
    "k_accum": {"bytes_per_unit": 236, "unit": "path ray folded"},
}


def dump_outputs(out_dir, mean, count):
    """Writes the framebuffer as DIR/mean.npy (H x W x 3) and DIR/count.npy (H x W), float32.  A frame above
    DUMP_LIMIT_BYTES is written as the same DUMP_SAMPLE_PIXELS pixels every run (seed 0, ascending row-major index in
    DIR/pixel_index.npy, float64): mean.npy is then N x 3 and count.npy N."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    h, w = count.shape
    arrays = {"mean": mean.astype(np.float32), "count": count.astype(np.float32)}
    if h*w*16 > DUMP_LIMIT_BYTES:
        idx = np.sort(np.random.default_rng(0).choice(h*w, DUMP_SAMPLE_PIXELS, replace=False))
        arrays = {"mean": arrays["mean"].reshape(h*w, 3)[idx], "count": arrays["count"].reshape(h*w)[idx],
                  "pixel_index": idx.astype(np.float64)}
    else:
        stale = os.path.join(out_dir, "pixel_index.npy")       # left by an earlier sampled dump into the same DIR
        if os.path.exists(stale):
            os.remove(stale)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def _measure(ctx, args, torch, dist, rank, world, local_rank, W, H, seed, steps, warmup, spp_per_step, e2e=True, keep_output=False):
    """Times `steps` steps of the hot path on this rank's tile share (device-resident), then the same through the host-buffer
    C-ABI call.  Returns a dict of raw numbers (rank-local + reduced); with keep_output, also the framebuffer after the
    timed steps (on rank 0: the whole frame)."""
    import numpy as np
    from tungsten_b200 import integrator
    all_tiles = integrator.dice_tiles(W, H, seed)
    my_tiles = integrator.shard_tiles(all_tiles, rank, world)
    shares = [integrator.shard_tiles(all_tiles, r, world) for r in range(world)] if world > 1 else [my_tiles]
    spp_step = spp_per_step*world
    stream = torch.cuda.current_stream()
    ctx.set_stream(stream.cuda_stream)              # renders, NCCL and the timing events share one stream
    if world > 1:
        max_pix = max(sum(t.w*t.h for t in sh) for sh in shares)
        send = torch.zeros(max_pix*3, dtype=torch.float32, device="cuda")
        recv = torch.zeros(world*max_pix*3, dtype=torch.float32, device="cuda")
    coll_events = []

    def step(i, resident=True, mean=None, count=None, time_collective=False):
        if resident:
            ctx.render_resident(spp_step, seed=seed, spp_begin=i*spp_step, tiles=my_tiles)
        else:
            ctx.render_tiles(spp_step, seed=seed, spp_begin=i*spp_step, tiles=my_tiles, mean=mean, count=count)
        if world > 1:
            if time_collective:
                e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True); e0.record(stream)
            ctx.pack_tiles(my_tiles, send.data_ptr())
            dist.all_gather_into_tensor(recv, send)
            if time_collective:
                e1.record(stream); coll_events.append((e0, e1))

    def timed(n_steps, first, resident, mean=None, count=None, time_collective=False):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ev0 = torch.cuda.Event(enable_timing=True); ev1 = torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        ev0.record(stream)
        for i in range(n_steps):
            step(first + i, resident, mean, count, time_collective)
        ev1.record(stream)
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        dev = ev0.elapsed_time(ev1)/1e3                       # CUDA events on the launching stream
        mine = dev
        if world > 1:
            tt = torch.tensor([dev], dtype=torch.float64, device="cuda")
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            dev = float(tt.item())
        return dev, mine, wall

    ctx.clear()
    for i in range(warmup):
        step(i)
    ctx.clear(); ctx.reset_stats(); ctx.set_profiling(True)
    stop = threading.Event(); clk = []
    th = threading.Thread(target=_clock_sampler, args=(stop, clk, local_rank), daemon=True); th.start()
    secs, my_secs, wall = timed(steps, 0, True, time_collective=True)
    stop.set(); th.join()
    st = ctx.stats()
    out = {"secs": secs, "wall": wall, "clk": clk, "spp_step": spp_step, "n_my_pix": sum(t.w*t.h for t in my_tiles), "st": st}
    if keep_output:
        if world > 1:                                 # the last all-gather holds every rank's share of the running mean
            ctx.clear()
            for r in range(world):
                ctx.unpack_tiles(shares[r], recv.data_ptr() + 4*r*max_pix*3, spp_step*steps)
        out["framebuffer"] = ctx.read_framebuffer()
    coll_ms = sum(a.elapsed_time(b) for a, b in coll_events)
    per_rank = [my_secs*1e3, st.total_ms, st.trace_ms, st.shadow_ms, coll_ms, float(st.samples)]
    if world > 1:
        tt = torch.tensor([float(st.samples), float(st.rays), float(st.hits), float(st.kernel_launches)], dtype=torch.float64, device="cuda")
        dist.all_reduce(tt)
        out["tot"] = [float(x) for x in tt.tolist()]
        pr = torch.tensor(per_rank, dtype=torch.float64, device="cuda"); allpr = torch.zeros(world*len(per_rank), dtype=torch.float64, device="cuda")
        dist.all_gather_into_tensor(allpr, pr)
        out["per_rank"] = allpr.view(world, len(per_rank)).cpu().tolist()
    else:
        out["tot"] = [float(st.samples), float(st.rays), float(st.hits), float(st.kernel_launches)]
        out["per_rank"] = [per_rank]

    # ---- N > 1: the gathered image is the one-rank image (de-tile every share, compare with rank 0 rendering everything alone)
    if world > 1:
        ctx.set_profiling(False)
        ctx.clear()
        step(0)
        torch.cuda.synchronize()
        for r in range(world):
            ctx.unpack_tiles(shares[r], recv.data_ptr() + 4*r*max_pix*3, spp_step)
        got, got_cnt = ctx.read_framebuffer()
        check = None
        if rank == 0:
            ctx.clear()
            ctx.render_resident(spp_step, seed=seed, spp_begin=0, tiles=all_tiles)
            want, want_cnt = ctx.read_framebuffer()
            check = {"equal": bool(np.array_equal(got, want) and np.array_equal(got_cnt, want_cnt)),
                     "what": "step 0 rendered by %d ranks, packed, all-gathered, unpacked on rank 0 vs the same %d spp of the whole frame rendered by rank 0 alone" % (world, spp_step),
                     "pixels": int(W*H), "max_abs_diff": float(np.abs(got - want).max())}
        out["gather_check"] = check

    # ---- end to end through the C ABI with host buffers ------------------------------------------
    if e2e:
        ctx.set_profiling(False)
        mean = np.zeros((H, W, 3), dtype=np.float32); count = np.zeros((H, W), dtype=np.uint32)
        e2e_steps = max(2, min(steps, 4))
        timed(1, 0, False, mean, count)
        mean[:] = 0; count[:] = 0
        ctx.reset_stats()
        e2e_secs, _, _ = timed(e2e_steps, 0, False, mean, count)
        e2e_samples = float(ctx.stats().samples)
        if world > 1:
            tt = torch.tensor([e2e_samples], dtype=torch.float64, device="cuda"); dist.all_reduce(tt); e2e_samples = float(tt.item())
        out["e2e"] = {"value": e2e_samples/e2e_secs/1e6, "unit": "Msamples/s", "h2d_bytes_per_step": W*H*16, "d2h_bytes_per_step": W*H*16,
                      "steps": e2e_steps}
    ctx.set_stream(None)
    return out


def _roofline(st, peak, peak_src, traffic):
    trace_gbs = (st.path_rays_traversed*ALG_BYTES_PER_QUERY/1e9)/(st.trace_ms/1e3) if st.trace_ms > 0 else 0.0
    shadow_gbs = (st.shadow_rays_traversed*ALG_BYTES_PER_QUERY/1e9)/(st.shadow_ms/1e3) if st.shadow_ms > 0 else 0.0
    queries_per_launch = st.path_rays_traversed/max(st.trace_launches, 1)
    r = {"bound": "hbm", "kernel": "k_trace (closest-hit traversal of path rays: 4-ary BVH, 64-byte quantised nodes)",
         "achieved": trace_gbs, "peak": peak, "unit": "GB/s", "frac": trace_gbs/peak,
         "traffic": traffic.get("dram_bytes_per_launch") if traffic else None,
         "traffic_over_algorithmic": (traffic["dram_bytes_per_launch"]/(traffic["queries_in_launch"]*ALG_BYTES_PER_QUERY)
                                      if traffic and traffic.get("queries_in_launch") else None),
         "traffic_source": traffic.get("source") if traffic else None,
         "peak_source": peak_src, "alg_bytes_per_query": ALG_BYTES_PER_QUERY,
         "queries": int(st.path_rays_traversed), "path_rays_total": int(st.path_rays), "kernel_ms": st.trace_ms, "launches": int(st.trace_launches),
         "alg_bytes_per_launch": queries_per_launch*ALG_BYTES_PER_QUERY,
         "mqueries_per_s": st.path_rays_traversed/st.trace_ms/1e3 if st.trace_ms > 0 else 0.0,
         "k_shadow": {"achieved": shadow_gbs, "frac": shadow_gbs/peak, "queries": int(st.shadow_rays_traversed), "shadow_rays_total": int(st.shadow_rays), "kernel_ms": st.shadow_ms,
                      "mqueries_per_s": st.shadow_rays_traversed/st.shadow_ms/1e3 if st.shadow_ms > 0 else 0.0},
         "note": "software BVH traversal is ALU-issue/latency bound with an L2-resident BVH (ncu: profiles/r02_*_k_trace*); 48 B/query is the algorithmic figure of SURVEY 8d"}
    units = {"k_regen": float(st.samples), "k_shade": float(st.path_rays), "k_accum": float(st.path_rays)}
    ms = {"k_regen": st.regen_ms, "k_shade": st.shade_ms, "k_accum": st.accum_ms}
    stream = {}
    for k, v in STREAM_BYTES.items():
        gbs = units[k]*v["bytes_per_unit"]/1e9/(ms[k]/1e3) if ms[k] > 0 else 0.0
        stream[k] = {"achieved": gbs, "frac": gbs/peak, "kernel_ms": ms[k], "bytes_per_unit": v["bytes_per_unit"], "unit_of_work": v["unit"], "units": units[k]}
    stream["note"] = ("bytes per unit are upper bounds of what the kernel moves for one unit (conditional records counted in full); ncu shows these kernels "
                      "issue bound, not DRAM bound (k_accum issues 0.74 inst/cycle/SMSP: 16-box BVH cut + analytic primitives per surviving ray)")
    other = {"k_shadow_prep_ms": st.prep_ms, "sort_ms": st.sort_ms, "iterations": int(st.iterations)}
    return r, stream, other


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=16)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--spp-per-step", type=int, default=64)
    ap.add_argument("--ref-spp", type=int, default=0, help="samples per pixel of one reference step (0 = calibrate to --ref-seconds)")
    ap.add_argument("--ref-seconds", type=float, default=6.0, help="target render time of one reference step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-other-configs", action="store_true", help="skip the short C2/C3/C4 measurements added to the C1 line")
    ap.add_argument("--config", default="c1", choices=sorted(CONFIGS))
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the framebuffer the last timed step left as DIR/<name>.npy (float32)")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    global W, H
    W, H = CONFIGS[args.config]["res"]
    if args.impl == "reference":
        if args.config == "c3":
            if rank == 0:
                print(json.dumps({"impl": "reference", "unavailable": "the stock reference cannot load mesh-instanced scenes from JSON (Instance::loadResources never loads its masters)"}))
            return
        return bench_reference(args, rank, world)

    import numpy as np
    import torch
    from tungsten_b200 import scene, lib
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the CUDA library is the only implementation")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def load(config):
        scene_path = make_scene(1024, config) if rank == 0 else None
        if world > 1:
            dist.barrier()
            scene_path = make_scene(1024, config)
        t0 = time.perf_counter()
        fs = scene.load_scene(scene_path)
        t1 = time.perf_counter()
        ctx = lib.Context(fs, device=local_rank)
        return scene_path, ctx, {"flatten_s": t1 - t0, "tgb200_create_s": time.perf_counter() - t1}

    seed = 0xBA5EBA11
    scene_path, ctx, build_times = load(args.config)
    info = ctx.scene_info()
    m = _measure(ctx, args, torch, dist, rank, world, local_rank, W, H, seed, args.steps, args.warmup, args.spp_per_step,
                 keep_output=args.dump_outputs is not None)
    if args.dump_outputs is not None and rank == 0:
        dump_outputs(args.dump_outputs, *m["framebuffer"])
    st = m["st"]
    tot_samples, tot_rays, tot_hits, tot_launches = m["tot"]
    value = tot_samples/m["secs"]/1e6
    peak, peak_src = hbm_peak()
    traffic = None
    tp = os.path.join(ROOT, "profiles", "k_trace_dram_bytes_per_launch.json")
    if os.path.exists(tp):
        try:
            traffic = json.load(open(tp))
        except Exception:
            traffic = None
    roof, stream, other = _roofline(st, peak, peak_src, traffic)
    ctx.close()

    # ---- the other BASELINE.json workloads, short runs on this GPU (one line per config is `bench.py --config cN`) -----------
    others = None
    if world == 1 and args.config == "c1" and not args.no_other_configs:
        others = {}
        for cfg in ("c2", "c3", "c4"):
            try:
                W, H = CONFIGS[cfg]["res"]
                _, c2, bt = load(cfg)
                i2 = c2.scene_info()
                mm = _measure(c2, args, torch, dist, rank, world, local_rank, W, H, seed, 3, 3, 8)
                s2 = mm["st"]
                others[cfg] = {"workload": CONFIGS[cfg]["label"], "value": mm["tot"][0]/mm["secs"]/1e6, "unit": "Msamples/s", "e2e": mm["e2e"]["value"],
                               "steps": 3, "warmup": 3, "spp_per_step": 8, "triangles": i2["n_tris"], "bvh_nodes": i2["n_nodes"],
                               "mrays_per_s": mm["tot"][1]/mm["secs"]/1e6,
                               "k_trace_mqueries_per_s": s2.path_rays_traversed/s2.trace_ms/1e3 if s2.trace_ms > 0 else 0.0,
                               "tgb200_create_s": bt["tgb200_create_s"]}
                c2.close()
            except Exception as e:                                   # a side measurement must not lose the headline line
                others[cfg] = {"error": str(e)[:200]}
        W, H = CONFIGS[args.config]["res"]

    if rank == 0:
        cpu = None
        if world == 1 and not args.no_cpu_baseline and args.config != "c3":
            host = host_cpu_info()
            cal = run_reference_binary(scene_path, 2, host["usable"])
            if cal is not None:
                spp_c = args.ref_spp if args.ref_spp > 0 else int(min(256, max(4, round(cal[0]*1e6*10.0/(W*H)))))
                r = run_reference_binary(scene_path, spp_c, host["usable"])
                if r is not None:
                    cpu = {"value": r[0], "unit": "Msamples/s", "cores": host["usable"], "kind": "reference",
                           "sample": "%d spp x %dx%d of the same scene rendered in %.2f s by oracle/_ref/tungsten -t %d ('Render time': excludes "
                                     "scene load + BVH build, as the GPU arm excludes tgb200_create)" % (spp_c, W, H, r[1], host["usable"]),
                           "host": host}
        pr = m["per_rank"]
        line = {
            "metric": "Msamples/sec (paths x spp)", "value": value, "unit": "Msamples/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3*m["secs"]/args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": CONFIGS[args.config]["label"],
                       "step": "%d spp of the frame per step (x%d steps = %d spp)" % (m["spp_step"], args.steps, m["spp_step"]*args.steps),
                       "tiles": "16x16, dealt to %d rank(s) in Morton order of the tile grid" % world, "paths_in_flight": info["capacity"],
                       "triangles": info["n_tris"], "bvh_nodes": info["n_nodes"], "geom_bytes": info["geom_bytes"],
                       "l2": "per-batch path state (%.0f MB) and geometry exceed the 126 MB L2; no explicit flush" % (info["capacity"]*344/1e6)},
            "timing": "CUDA events on the stream the kernels (and the all-gather) are launched on, max over ranks; wall clock of the same region %.3f s" % m["wall"],
            "mrays_per_s": tot_rays/m["secs"]/1e6, "mray_hits_per_s": tot_hits/m["secs"]/1e6,
            "device_ms": max(p[1] for p in pr), "gpu_launches": int(tot_launches),
            "ranks": {"step_ms_min": min(p[0] for p in pr)/args.steps, "step_ms_max": max(p[0] for p in pr)/args.steps,
                      "device_ms_min": min(p[1] for p in pr), "device_ms_max": max(p[1] for p in pr),
                      "k_trace_ms_min": min(p[2] for p in pr), "k_trace_ms_max": max(p[2] for p in pr),
                      "collective_ms_per_step_max": max(p[4] for p in pr)/args.steps,
                      "samples_min": min(p[5] for p in pr), "samples_max": max(p[5] for p in pr)},
            "gather_check": m.get("gather_check"),
            "e2e": m["e2e"],
            "roofline": roof, "roofline_streaming": stream, "loop": other,
            "setup": dict(build_times, note="scene flattening and tgb200_create (host SAH build of the BVH + upload) are outside the timed region, as the "
                                            "reference's 'Render time' excludes its scene load and Embree build"),
            "other_configs": others,
            "cpu_baseline": cpu,
            "clocks": _summarise_clocks(m["clk"]),
        }
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
