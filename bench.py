#!/usr/bin/env python
"""bench.py — BASELINE.json metric: EKF-SLAM frames/sec @320x240, N = 100 features (config C4:
n = 313, m = 200, 11x11 patch, +-20 px search ellipse), aggregate over independent camera streams.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--streams B] [--impl ours|reference] [--dump-outputs DIR]

A "step" = one GoOneStep pass (predict -> select -> patch search -> EKF update -> normalise ->
cull -> symmetrise) of every camera stream resident on the GPU over one new frame each.
`value`  : frames/s with the frames already resident in HBM (frame ring), CUDA-event timed.
`e2e`    : the same metric through the C-ABI call sl2_step_host with HOST (pinned) frames in and
           camera states out, host<->device copies inside the timed region.
Multi-GPU: replicas only (independent camera sequences, no collective on the data path); the
barrier + max-over-ranks timing uses torch.distributed (NCCL).
`--impl reference`: the CPU oracle (a port: the reference cannot be built here) on all host cores.
`--dump-outputs DIR`: after the timed steps of the main workload, what they computed (see dump_outputs) as
           DIR/<name>.npy, so that two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "EKF-SLAM frames/sec @320x240 N=100 feats"
UNIT = "frames/s"
WORKLOAD = "C4: synthetic 320x240, 100 features, EKF state dim 313, 11x11 patch, +-20px ellipse"
WORKLOADS = {"C1": "C1: synthetic 320x240, 4 known + 16 features, 10 selected per frame, ellipses from S_i",
             "C2": "C2: synthetic 320x240, 50 features, 11x11 patch, +-20px ellipse",
             "C3": "C3: synthetic 640x480, 100 features, 15x15 patch, +-40px ellipse", "C4": WORKLOAD}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--streams", type=int, default=296, help="camera streams per GPU")
    ap.add_argument("--config", default="C4")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--ring", type=int, default=4, help="distinct frames per stream")
    ap.add_argument("--unique", type=int, default=16, help="distinct synthetic scenes (tiled over streams)")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="CPU baseline sample budget")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dist-selftest", action="store_true", help="CPU/gloo check of the N>1 plumbing")
    ap.add_argument("--cpu-threads", type=int, default=0, help="host threads of the CPU legs (0 = all)")
    ap.add_argument("--only-main", action="store_true", help="skip the legs of the other configs / single stream")
    ap.add_argument("--step-groups", type=int, default=1, choices=[1, 2],
                    help="staggered stream groups of the fused step (1 = serial kernel order)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the states / feature results of the last timed step as DIR/<name>.npy")
    return ap.parse_args()


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)), "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}, "fallback"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.rows = []
        self.stop_flag = threading.Event()

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                      "--format=csv,noheader,nounits"], capture_output=True,
                                     text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self.stop_flag.wait(0.2)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[2 + i] == "Active" for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None,
                "sm_max_mhz": float(self.rows[0][1]) if self.rows[0][1].replace(".", "").isdigit() else None,
                "reasons": reasons}


def make_scenes(name, unique, ring, base_stream=0):
    from scenelib2_b200 import synth
    return [synth.make_scene(name, stream_id=base_stream + i, n_frames=ring) for i in range(unique)]


def oracle_slams(po, scenes, count):
    slams = []
    for i in range(count):
        sc = scenes[i % len(scenes)]
        cfg = po.make_config(width=sc.width, height=sc.height, fku=sc.cam8[2], fkv=sc.cam8[3],
                             u0=sc.cam8[4], v0=sc.cam8[5], kd1=sc.cam8[6], sd=sc.cam8[7],
                             delta_t=sc.delta_t, n_select=sc.n_select, boxsize=sc.boxsize,
                             search_override=sc.search_override)
        s = po.Slam(cfg)
        for k in range(sc.n_features):
            s.add_feature(sc.x0[13 + 3 * k:16 + 3 * k], sc.xp_org[k], sc.patches[k])
        s.set_state(sc.x0, sc.P0)
        slams.append(s)
    return slams


def cpu_run(scenes, seconds, threads=None, pin=True):
    """Oracle (CPU port of the reference path) timed on the host cores over a bounded sample: one independent
    camera stream per thread, each thread pinned to its own usable CPU (affinity mask capped by the cgroup quota)."""
    from oracle import pyoracle as po
    po.build()
    threads = threads or po.usable_cpus() or 1
    slams = oracle_slams(po, scenes, threads)
    frames = [scenes[i % len(scenes)].frames for i in range(threads)]
    t1, _ = po.run_slams_pinned(slams, frames, 1, threads, pin)   # calibration (also warms caches)
    steps = max(2, int(seconds / max(t1, 1e-3)))
    t, gs = po.run_slams_pinned(slams, frames, steps, threads, pin)
    fps = threads * steps / t
    # "dense-resident" variant of SURVEY 8(d): the same run without the reference's 4 gather / scatter passes per
    # frame (monoslam.cpp:518-614), whose time the oracle measures per stream; gs is summed over the streams
    gs_share = gs / max(threads * t, 1e-12)
    return {"fps": fps, "threads": threads, "steps": steps, "seconds": t, "gather_scatter_share": gs_share,
            "fps_dense_resident": fps / max(1e-9, 1.0 - gs_share)}


def cpu_baseline_block(scenes, seconds, threads=None):
    """cpu_baseline object: all usable cores (the headline), plus 1 and 8 threads of the same sample."""
    from oracle import pyoracle as po
    po.build()
    usable = threads or po.usable_cpus() or 1
    legs = {}
    for nt, share in ((1, 0.2), (min(8, usable), 0.25), (usable, 0.55)):
        if nt in legs:
            continue
        legs[nt] = cpu_run(scenes, seconds * share, nt)
    full = legs[usable]
    return {"value": full["fps"], "unit": UNIT, "cores": usable, "kind": "port",
            "sample": "%d streams (1 per pinned thread) x %d oracle steps (%.1f s)" % (usable, full["steps"], full["seconds"]),
            "frames_per_s_per_core": full["fps"] / usable,
            "by_threads": {str(k): round(v["fps"], 2) for k, v in sorted(legs.items())},
            "hardware_threads_of_the_box": po.hardware_threads(),
            "cores_how": "min(sched_getaffinity, cgroup cpu.max quota)",
            "storage": "faithful (per-feature heap blocks + 4 gather/scatter passes per frame, like the reference)",
            "gather_scatter_share": round(full["gather_scatter_share"], 4),
            "dense_resident_value": full["fps_dense_resident"],
            "dense_resident_how": "same run minus the measured time of the gather/scatter passes (monoslam.cpp:518-614)"}


def dist_selftest(rank, world):
    """gloo on CPU: the same barrier / MAX-reduce / per-rank stream bases the GPU run uses."""
    import torch
    import torch.distributed as dist
    dist.init_process_group("gloo")
    dist.barrier()
    t = torch.tensor([10.0 * (rank + 1)])
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    n = torch.tensor([3.0])
    dist.all_reduce(n, op=dist.ReduceOp.SUM)
    bases = [None] * world
    dist.all_gather_object(bases, rank * 1000)
    if rank == 0:
        print(json.dumps({"world": world, "max_ms": float(t.item()), "sum_streams": int(n.item()),
                          "stream_bases": bases}))
    dist.destroy_process_group()


def reference_sources_rate(config, seconds=3.0):
    """frames/s of the reference's own MonoSLAM::GoOneStep (oracle/_ref/libsl2refmodels.so), one thread."""
    try:
        import tempfile
        from oracle import pyoracle as po
        from scenelib2_b200 import synth
        if po.ref_models() is None:
            return None
        sc = synth.make_scene(config, n_frames=4, override=False)
        r = po.RefSlam(sc, tempfile.mkdtemp(prefix="sl2ref_"))
        t0, n = time.time(), 0
        while time.time() - t0 < seconds:
            r.step(sc.frames[n % 4])
            n += 1
        return {"value": n / (time.time() - t0), "unit": UNIT, "cores": 1, "sample": "%d steps" % n,
                "workload": "same scene, search ellipses from the EKF's own S_i"}
    except Exception as e:  # informational only
        return {"unavailable": str(e)[:120]}


def run_reference(args, rank, world):
    if rank != 0:
        return
    from oracle import pyoracle as po
    po.build()
    scenes = make_scenes(args.config, min(args.unique, 8), args.ring)
    budget = args.cpu_seconds if args.cpu_seconds < 12.0 else max(2.0, min(40.0, 120.0 / max(1, args.steps + args.warmup)))
    vals, last = [], None
    threads = args.cpu_threads or po.usable_cpus() or 1
    for k in range(args.warmup + args.steps):
        last = cpu_run(scenes, budget, threads)
        if k >= args.warmup:
            vals.append(last["fps"])
    v = float(np.mean(vals))
    sample = "%d streams (1 per pinned thread) x ~%.0f s of oracle steps per bench step" % (threads, budget)
    ref_src = reference_sources_rate(args.config)
    one = cpu_run(scenes, min(3.0, budget), 1)
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus,
        "steps": len(vals), "warmup": args.warmup, "ms_per_step": 1e3 * threads / v,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic", "config": {"workload": WORKLOADS.get(args.config, WORKLOAD), "streams": threads,
                                        "note": "CPU oracle = port of the reference path (Eigen3/OpenCV absent: "
                                                "the reference binary cannot be built); faithful block storage",
                                        # for information: the reference's OWN tracking sources compiled against
                                        # stand-ins for Eigen/OpenCV/Pangolin (oracle/_ref/libsl2refmodels.so), one
                                        # thread, ellipses from S_i (it has no fixed-ellipse switch).  Slower than the
                                        # port (its matrix stand-in is not Eigen), so the port stays the baseline.
                                        "reference_sources_with_standins": ref_src},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample,
                         "frames_per_s_per_core": v / threads, "one_thread_value": one["fps"],
                         "hardware_threads_of_the_box": po.hardware_threads(),
                         "cores_how": "min(sched_getaffinity, cgroup cpu.max quota), one pinned thread per core",
                         "gather_scatter_share": round(last["gather_scatter_share"], 4),
                         "dense_resident_value": v / max(1e-9, 1.0 - last["gather_scatter_share"])},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def _traffic(config, kernel, B):
    """dram__bytes_read + write per launch of `kernel`, from the ncu capture of THIS config (per stream x B), or None
    when no capture of that config is committed (profiles/r02_dram_bytes.json, written by tools/ncu_traffic.py)."""
    fp = os.path.join(ROOT, "profiles", "r02_dram_bytes.json")
    if not os.path.exists(fp):
        return None
    try:
        v = json.load(open(fp)).get(config, {}).get(kernel)
        return None if v is None else v["bytes_per_stream"] * B
    except Exception:
        return None


DUMP_COV_STREAMS = 16


def dump_outputs(ctx, B, directory):
    """What a caller of the step receives for every stream -- state x, covariance diagonal, per-feature results --
    padded with NaN to the largest state / feature count, and the full covariance of a fixed, seeded sample of
    DUMP_COV_STREAMS streams (all of them would exceed 64 MB at the C4 size).  float64 throughout."""
    os.makedirs(directory, exist_ok=True)
    nf = np.array([ctx.num_features(s) for s in range(B)])
    n = 13 + 3 * int(nf.max())
    N = int(nf.max())
    pick = np.sort(np.random.default_rng(0).choice(B, min(B, DUMP_COV_STREAMS), replace=False))
    out = {"num_features": nf.astype(np.float64), "state_x": np.full((B, n), np.nan),
           "state_cov_diag": np.full((B, n), np.nan), "state_cov_streams": pick.astype(np.float64),
           "state_cov": np.full((len(pick), n, n), np.nan)}
    widths = {"h": 2, "z": 2, "S": 4, "flags": 1, "attempted": 1, "successful": 1, "select_rank": 1}
    for k, w in widths.items():
        out["feature_" + k] = np.full((B, N, w), np.nan)
    for s in range(B):
        x, P = ctx.get_state(s)
        out["state_x"][s, :len(x)] = x
        out["state_cov_diag"][s, :len(x)] = np.diag(P)
        if s in pick:
            out["state_cov"][np.searchsorted(pick, s), :len(x), :len(x)] = P
        for k, v in ctx.features(s).items():
            out["feature_" + k][s, :len(v)] = np.asarray(v, np.float64).reshape(len(v), widths[k])
    for k, v in out.items():
        np.save(os.path.join(directory, k + ".npy"), v)


def measure_config(args, config, B, steps, warmup, rank, local_rank, world, stream, dev, e2e=True, clocks=False,
                   dump=None):
    """One workload (BASELINE config) on this rank's GPU: device-resident throughput, end-to-end throughput through
    the C ABI with host frames, per-kernel times.  Returns a dict (times already MAX-reduced over ranks)."""
    import torch
    import torch.distributed as dist
    import scenelib2_b200 as sl2
    from scenelib2_b200 import synth

    R = args.ring
    scenes = make_scenes(config, min(args.unique, B), R, base_stream=rank * 1000)
    sc0 = scenes[0]
    N, n, H, W = sc0.n_features, sc0.n, sc0.height, sc0.width
    cfg = sl2.config_for_scene(sc0, num_streams=B, frame_slots=R, device=local_rank,
                               cuda_stream=stream.cuda_stream)
    ctx = sl2.Context(cfg)
    ctx.set_step_groups(args.step_groups)
    for s in range(B):
        sl2.load_scene(ctx, s, scenes[s % len(scenes)])
    host = torch.empty((R, B, H, W), dtype=torch.uint8, pin_memory=True)   # pinned host frame ring
    hv = host.numpy()
    for s in range(B):
        hv[:, s] = scenes[s % len(scenes)].frames
    for k in range(R):
        ctx.set_frames_ptr(k, host[k].data_ptr())
    xv_out = torch.empty((R, B, 13), dtype=torch.float64, pin_memory=True)
    ctx.sync()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, nsteps, post=None):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record(stream)
        for k in range(nsteps):
            fn(k)
        if post:
            post()
        e1.record(stream)
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    out = {"config": config, "workload": WORKLOADS.get(config, config), "streams_per_gpu": B, "state_dim": n,
           "features": N, "frame": [W, H]}
    # ---- device-resident leg (`value`) ----------------------------------------------------------
    for k in range(warmup):
        ctx.step(k % R)
    sampler = None
    if clocks:
        sampler = ClockSampler(local_rank)
        sampler.start()
    l0 = ctx.launch_count()
    ms = timed(lambda k: ctx.step(k % R), steps, post=ctx.join)
    out["gpu_launches"] = int(ctx.launch_count() - l0)
    if sampler:
        sampler.stop_flag.set()
        sampler.join(timeout=2)
        out["clocks"] = sampler.summary()
    out["ms_per_step"] = ms / steps
    out["value"] = world * B * steps / (ms * 1e-3)
    if dump:
        dump_outputs(ctx, B, dump)

    # ---- per-kernel durations (CUDA events on the launching stream, one sync per step) ----------
    ctx.enable_timing(True)
    kt, ku = np.zeros(4), np.zeros(5)
    for k in range(steps):
        ctx.step(k % R)
        kt += ctx.last_step_times()
        ku += ctx.last_update_times()
    kt /= steps
    ku /= steps
    ctx.enable_timing(False)
    out["kernel_ms"] = {"predict_select": float(kt[0]), "patch_search": float(kt[1]), "ekf_update": float(kt[2]),
                        "cull": float(kt[3]),
                        "ekf_update_kernels": {"hp": float(ku[0]), "chol": float(ku[1]), "solve": float(ku[2]),
                                               "syrk": float(ku[3]), "finish": float(ku[4])}}

    # ---- end-to-end leg: host frames in, camera states out, through the C ABI -----------------
    # every step: pinned host frames -> H2D -> GoOneStep of all streams -> D2H of the camera states;
    # the copy of step t+1 overlaps the kernels of step t (frame ring); the region ends when the
    # last result has landed in host memory (ctx.sync).
    if e2e:
        def e2e_step(k):
            ctx.step_host_async(k % R, host[k % R].data_ptr(), xv_out[k % R].data_ptr())
        for k in range(min(3, warmup)):
            e2e_step(k)
        ctx.sync()
        ms_e2e = timed(e2e_step, steps, post=ctx.sync)
        ms_sync = timed(lambda k: ctx.step_host(k % R, host[k % R].data_ptr(), xv_out[k % R].data_ptr()),
                        max(3, steps // 4))
        out["e2e"] = {"value": world * B * steps / (ms_e2e * 1e-3), "unit": UNIT, "h2d_bytes_per_step": world * B * H * W,
                      "d2h_bytes_per_step": world * B * 13 * 8, "ms_per_step": ms_e2e / steps,
                      "api": "sl2_step_host_async over a ring of %d pinned frame sets" % R,
                      "blocking_call_value": world * B * max(3, steps // 4) / (ms_sync * 1e-3)}
    out["matched_fraction"] = float(np.mean([(ctx.features(s)["flags"] & 2).astype(bool).mean()
                                             for s in sorted({0, B // 2, B - 1})]))
    out["features_left_stream0"] = ctx.num_features(0)

    # ---- rooflines ------------------------------------------------------------------------------
    pk, pk_kind = peaks()
    rad = sc0.meta["config"]["radius"] or 20   # C1: ellipses come from S_i; 20 px = the tile radius
    nsel = min(sc0.n_select, N)
    search_bytes = B * nsel * synth.algorithmic_search_bytes(sc0.boxsize, rad)   # per launch (SURVEY 8(d))
    ach = search_bytes / (kt[1] * 1e-3) / 1e9
    m = 2 * nsel
    flops = synth.ekf_structured_flops(n, m) * B
    fp64_peak, fp64_kind = 37.0, "nominal"
    fp = os.path.join(ROOT, "profiles", "fp64_peak_measured.json")
    if os.path.exists(fp):
        fp64_peak, fp64_kind = json.load(open(fp))["fp64_tflops"], "measured (tools/fp64_pipes.cu)"
    upd_tr = [_traffic(config, k, B) for k in ("upd_hp", "upd_chol", "upd_solve", "upd_syrk", "upd_finish")]
    out["roofline"] = {
        "kernel": "EKF update = upd_hp + upd_chol + upd_solve + upd_syrk + upd_finish (%.0f %% of the step)"
                  % (100 * kt[2] / kt.sum()),
        "bound": "tensor", "achieved": flops / (kt[2] * 1e-3) / 1e12, "peak": fp64_peak, "unit": "TFLOP/s",
        "frac": flops / (kt[2] * 1e-3) / 1e12 / fp64_peak,
        "traffic": None if any(v is None for v in upd_tr) else float(sum(upd_tr)), "peak_kind": fp64_kind,
        "algorithmic_flops_per_launch": flops, "kernel_ms": float(kt[2]),
        "note": "FP64 DMMA m8n8k4 (tcgen05 has no FP64 kind); structured-minimum FLOPs of SURVEY 8(d) over the "
                "summed duration of the five update kernels"}
    out["roofline_patch_search"] = {
        "kernel": "search_kernel (patch search)", "bound": "hbm", "achieved": ach, "peak": pk["hbm_gbs"],
        "unit": "GB/s", "frac": ach / pk["hbm_gbs"], "traffic": _traffic(config, "search", B), "peak_kind": pk_kind,
        "algorithmic_bytes_per_launch": search_bytes, "kernel_ms": float(kt[1]),
        "note": "integer / FP64 issue bound, not HBM bound: see DESIGN.md 3.1"}
    ctx.close()
    return out, scenes


def shim_rate(config, repeat=60):
    """frames/s a SceneLib2 CALLER sees: the reference-shaped C++ class surface (scenelib2_b200/host) driven like
    examples/MonoSlamSceneLib1.cpp by sl2_headless -- ONE camera stream, GoOneStep per frame with the frame upload
    and the refresh of every host mirror (Feature::y_/Pxy_/Pyy_/matrix_block_list_) inside the timed region."""
    import tempfile
    from scenelib2_b200 import synth
    exe = os.path.join(ROOT, "scenelib2_b200", "host", "sl2_headless")
    if not os.path.exists(exe):
        return {"unavailable": "sl2_headless not built"}
    try:
        kw = {}
        if config == "C1":
            kp = os.path.join(ROOT, "tests", "golden", "known_patches.npy")
            if os.path.exists(kp):
                kw["known_patches"] = np.load(kp)
        sc = synth.make_scene(config, n_frames=4, **kw)
        d = tempfile.mkdtemp(prefix="sl2shim_")
        Pxx = np.diag([4e-4] * 3 + [2e-5] * 4 + [1e-3] * 3 + [1e-3] * 3)   # cf. data/SceneLib2.cfg:85-115
        cfg = synth.write_reference_case(d, sc, Pxx)
        env = dict(os.environ, SL2_HEADLESS_REPEAT=str(repeat))
        r = subprocess.run([exe, cfg, os.path.join(d, "frames.raw"), str(sc.width), str(sc.height), "4"],
                           capture_output=True, text=True, env=env, timeout=120)
        for ln in r.stdout.splitlines():
            if ln.startswith("shim_frames_per_s"):
                t = ln.split()
                return {"value": float(t[1]), "unit": UNIT, "streams": 1, "features": int(t[5]),
                        "api": "SceneLib2::MonoSLAM::GoOneStep of the host shim (full host mirrors per frame)"}
        return {"unavailable": (r.stderr or r.stdout)[-160:]}
    except Exception as e:   # informational leg
        return {"unavailable": str(e)[:160]}


def aux_rates():
    """Rows N2 / N3 of SURVEY 8(f) through the public API (host buffers in, results out, one call = one H2D, the
    kernels, one D2H): the Shi-Tomasi detector over the reference's 80x60 initialisation window
    (monoslam.cpp:947-948), batches of such windows and a whole frame; and the partially-initialised-feature cycle
    (particle prediction, overlapping-ellipse search, re-weighting) for 1 and 8 features of 100 particles.  The
    oracle port is timed on the same inputs (one host core)."""
    import scenelib2_b200 as sl2
    from scenelib2_b200 import synth
    from oracle import pyoracle as po
    out = {}
    try:
        rng = np.random.default_rng(5)
        img = synth.make_texture(rng, 240, 320)
        cfg = sl2.default_config()
        cfg.width, cfg.height, cfg.boxsize, cfg.max_features = 320, 240, 11, 4
        ctx = sl2.Context(cfg)
        ctx.set_features(0, np.zeros((1, 3)), np.tile([0, 0, 0, 1, 0, 0, 0.0], (1, 1)), np.zeros((1, 11, 11), np.uint8))
        ctx.set_frame(0, 0, img)

        def rate(regions, reps=30):
            for _ in range(3):
                ctx.find_best_patch(0, 0, regions)
            t0 = time.perf_counter()
            for _ in range(reps):
                ctx.find_best_patch(0, 0, regions)
            return (time.perf_counter() - t0) / reps

        one = np.array([[120, 90, 200, 150]], np.int32)
        x0 = rng.integers(6, 234, 64)
        y0 = rng.integers(6, 174, 64)
        many = np.column_stack([x0, y0, x0 + 80, y0 + 60]).astype(np.int32)
        full = np.array([[0, 0, 320, 240]], np.int32)
        t1, t64, tf = rate(one), rate(many), rate(full)
        c0 = time.perf_counter()
        creps = 20
        for _ in range(creps):
            po.find_best_patch(img, 11, one[0])
        tc = (time.perf_counter() - c0) / creps
        out["N3_detector"] = {
            "workload": "Shi-Tomasi best patch, 11x11 box, 320x240 frame; window = 80x60 (monoslam.cpp:947-948)",
            "api": "sl2_find_best_patch (blocking: regions H2D, 2 kernels, results D2H)",
            "us_per_call_1_window": t1 * 1e6, "us_per_call_64_windows": t64 * 1e6, "us_per_window_batched": t64 / 64 * 1e6,
            "us_per_call_full_frame": tf * 1e6, "positions_per_s_batched": 64 * 80 * 60 / t64,
            "cpu_port_us_per_window": tc * 1e6, "cpu_cores": 1}
        ctx.close()
    except Exception as e:   # informational leg
        out["N3_detector"] = {"unavailable": str(e)[:160]}
    try:
        rng = np.random.default_rng(6)
        img = synth.make_texture(rng, 240, 320)
        cfg = sl2.default_config()
        cfg.width, cfg.height, cfg.boxsize, cfg.max_features = 320, 240, 11, 4
        ctx = sl2.Context(cfg)
        ctx.set_features(0, np.zeros((1, 3)), np.tile([0, 0, 0, 1, 0, 0, 0.0], (1, 1)), np.zeros((1, 11, 11), np.uint8))
        ctx.set_frame(0, 0, img)
        cam8 = np.array([cfg.width, cfg.height, cfg.fku, cfg.fkv, cfg.u0, cfg.v0, cfg.kd1, cfg.sd], float)
        xv = np.zeros(13)
        xv[:3] = [0.06, -0.03, 0.01]
        xv[3:7] = np.array([1.0, 0.01, -0.02, 0.015]) / np.linalg.norm([1.0, 0.01, -0.02, 0.015])
        A = rng.normal(0, 1, (16, 16))
        P = A @ A.T * 2e-6 + 1e-8 * np.eye(16)
        ctx.set_state(0, np.concatenate([xv, [0.1, 0.1, 2.0]]), P)
        F, K = 8, 100   # kNumberOfParticles-sized features (monoslam.cpp: 100 depth hypotheses 0.5 .. 5 m)
        ypi, Pxy, Pyy = np.zeros((F, 6)), np.zeros((F, 13, 6)), np.zeros((F, 6, 6))
        lam = np.tile(np.linspace(0.5, 5.0, K), (F, 1))
        prob = np.full((F, K), 1.0 / K)
        patches = np.zeros((F, 11, 11), np.uint8)
        for f in range(F):
            u, v = rng.uniform(60, 260), rng.uniform(50, 190)
            hh = np.array([-(u - cfg.u0) / cfg.fku, -(v - cfg.v0) / cfg.fkv, 1.0])
            ypi[f, 3:] = hh / np.linalg.norm(hh)
            Af = rng.normal(0, 1, (19, 19))
            Pf = Af @ Af.T * 2e-6 + 1e-8 * np.eye(19)
            Pxy[f], Pyy[f] = Pf[:13, 13:], Pf[13:, 13:]
            hm = po.predict_particles(cam8, xv, ypi[f], [2.0], P[:13, :13], Pxy[f], Pyy[f])[0][0]
            cu, cv = int(round(hm[0])), int(round(hm[1]))
            patches[f] = img[cv - 5:cv + 6, cu - 5:cu + 6]

        def rate(nf, reps=30):
            for _ in range(3):
                ctx.measure_partial_features(0, 0, patches[:nf], ypi[:nf], Pxy[:nf], Pyy[:nf], lam[:nf], 0.05, prob[:nf])
            t0 = time.perf_counter()
            for _ in range(reps):
                ctx.measure_partial_features(0, 0, patches[:nf], ypi[:nf], Pxy[:nf], Pyy[:nf], lam[:nf], 0.05, prob[:nf])
            return (time.perf_counter() - t0) / reps

        t1, t8 = rate(1), rate(F)
        c0 = time.perf_counter()
        creps = 3
        for _ in range(creps):
            oh, _, osi, odet = po.predict_particles(cam8, xv, ypi[0], lam[0], P[:13, :13], Pxy[0], Pyy[0])
            ou, ov, of, _ = po.smoe_search(img, patches[0], osi, oh)
            po.particle_update(oh, osi, odet, lam[0], np.column_stack([ou, ov]), of, 0.05, prob[0])
        tc = (time.perf_counter() - c0) / creps
        out["N2_partial_features"] = {
            "workload": "partially-initialised features, 100 depth particles each, 11x11 template, 320x240 frame: "
                        "ellipse prediction + overlapping-ellipse search + particle re-weighting (monoslam.cpp:1347-1493)",
            "api": "sl2_measure_partial_features (blocking: one H2D, 4 kernels, one D2H for all features of the call)",
            "us_per_call_1_feature": t1 * 1e6, "us_per_call_8_features": t8 * 1e6, "us_per_feature_batched": t8 / F * 1e6,
            "cpu_port_us_per_feature": tc * 1e6, "cpu_cores": 1}
        ctx.close()
    except Exception as e:   # informational leg
        out["N2_partial_features"] = {"unavailable": str(e)[:160]}
    return out


def run_ours(args, rank, local_rank, world):
    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl ours needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    # a dedicated (non-default) torch stream: the library launches on it, torch events time it
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)

    B = args.streams
    main, scenes = measure_config(args, args.config, B, args.steps, args.warmup, rank, local_rank, world, stream, dev,
                                  clocks=True, dump=args.dump_outputs if rank == 0 else None)
    # the other BASELINE configs (north star: N in {20, 50, 100}; C3 on 8 GPUs = C5) and the single-stream latency
    extra = {}
    if not args.only_main:
        short = max(5, min(args.steps, 20))
        for cname in ("C1", "C2", "C3", "C4"):
            if cname == args.config:
                continue
            r, _ = measure_config(args, cname, B, short, 3, rank, local_rank, world, stream, dev)
            key = "C5" if (cname == "C3" and world == 8) else cname
            if key == "C5":
                r["workload"] = "C5: 8 independent synthetic 640x480 stream sets, 100 features each, one set per GPU"
            extra[key] = {k: r[k] for k in ("workload", "streams_per_gpu", "state_dim", "value", "ms_per_step", "e2e",
                                            "kernel_ms", "roofline", "roofline_patch_search", "matched_fraction",
                                            "gpu_launches")}
        one, _ = measure_config(args, args.config, 1, short, 3, rank, local_rank, world, stream, dev, e2e=False)
        extra["single_stream"] = {"workload": one["workload"] + ", ONE camera stream per GPU (latency)",
                                  "ms_per_frame": one["ms_per_step"], "value": one["value"],
                                  "kernel_ms": one["kernel_ms"]}
        if rank == 0:
            extra["shim_single_stream"] = {c: shim_rate(c) for c in ("C1", "C4")}
            extra.update(aux_rates())

    if rank == 0:
        sc0 = scenes[0]
        line = {
            "metric": METRIC, "value": main["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": main["ms_per_step"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64 (EKF, scores) + u8/int32 (correlation sums)",
            "data": "synthetic",
            "config": {"workload": main["workload"], "streams_per_gpu": B, "frames_per_step": B * world,
                       "state_dim": main["state_dim"], "measurements": 2 * min(sc0.n_select, sc0.n_features),
                       "parallelism": "replicas x%d (no collective)" % world,
                       "l2": "per-step working set %.0f MB (P + scratch + frames of %d streams) exceeds the 126 MB L2"
                             % ((B * (sc0.n_features * 3 + 13) ** 2 * 8 * 2.1) / 1e6, B),
                       "matched_fraction": main["matched_fraction"], "features_left_stream0": main["features_left_stream0"],
                       "step_groups": args.step_groups,
                       "kernel_timing": "kernel_ms / roofline: separate pass in serial kernel order (whole batch per "
                                        "launch, CUDA events between launches); the timed `value` and `e2e` regions "
                                        "launch back to back"},
            "e2e": main["e2e"], "gpu_launches": main["gpu_launches"], "clocks": main.get("clocks"),
            # the step's dominant stage = the EKF update (five kernels on the FP64 tensor path); MEASURED_PEAKS.json
            # has no FP64 entry, so the peak is the DMMA rate measured on this pool by tools/fp64_pipes.cu
            "roofline": main["roofline"],
            # the metric also asks for the patch search against the HBM roofline
            "roofline_patch_search": main["roofline_patch_search"],
            "kernel_ms": main["kernel_ms"],
            "configs": extra,
        }
        if not args.no_cpu_baseline and world == 1:
            line["cpu_baseline"] = cpu_baseline_block(scenes, args.cpu_seconds, args.cpu_threads or None)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    a = parse()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if a.dist_selftest:
        dist_selftest(rank, world)
    elif a.impl == "reference":
        if a.dump_outputs:
            raise SystemExit("--dump-outputs writes the outputs of --impl ours")
        run_reference(a, rank, world)
    else:
        run_ours(a, rank, local_rank, world)
