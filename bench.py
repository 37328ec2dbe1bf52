#!/usr/bin/env python
"""bench.py — Mpixels/s of the feature-detection hot path on synthetic frames.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B] [--workload W] [--impl reference] [--dump-outputs DIR]
  torchrun --nproc-per-node N bench.py --gpus N ...        (one rank per GPU, frames sharded, no
                                                            data-path collective: weak scaling)

Workloads (BASELINE.json):
  composite (default)  Harris + Canny + FHOG on B 3840x2160 frames per GPU per step (the metric's configuration)
  surf                 SURF key points + descriptors on B 3840x2160 frames per GPU per step (config 4: 64 per GPU)
  stream8k             Harris + Canny on B 7680x4320 grey frames per GPU per step (config 5)
A step = one pass of the workload's detectors over the batch.  The JSON line reports
  value   : whole-job Mpixels/s with the frames already resident in HBM (device-timed, CUDA events)
  e2e     : the same through the public host API (pinned host buffers, H2D + D2H inside the timing)
  roofline: the fused Harris gradient+response kernel (composite, stream8k), algorithmic 5 B/pixel (u8 in, f32 R out),
            achieved GB/s from CUDA events around back-to-back launches, against MEASURED_PEAKS.json
  cpu_baseline: the reference's own C/C++ (oracle/_ref) on this box's host cores, bounded sample.
The Harris path timed here is the default, certified one: its corner lists and strengths are the reference's bit for bit.
`--impl reference` times only the reference CPU implementation (all host threads) on the same workload.
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

HARRIS_KW = dict(k=0.06, sigma_d=1.0, sigma_i=2.5, threshold=130.0, gaussian=0, gradient=0, measure=0)
CANNY_KW = dict(s=2.0, low_thr=3.0, high_thr=10.0, accGrad=True)
FHOG_KW = dict(cell=8, frp=1, fcp=1)
SURF_KW = dict(max_points=10000, detection_threshold=30.0)

WORKLOADS = {
    "composite": dict(nx=3840, ny=2160, dets=["harris", "canny", "fhog"], name="harris+canny+fhog @3840x2160",
                      metric="Mpixels/sec (Harris+Canny+HOG) at 4K frames", batch=16),
    "surf": dict(nx=3840, ny=2160, dets=["surf"], name="surf @3840x2160 (max_points=10000, detection_threshold=30)",
                 metric="Mpixels/sec (SURF key points + descriptors) at 4K frames", batch=16),
    "stream8k": dict(nx=7680, ny=4320, dets=["harris", "canny"], name="harris+canny @7680x4320",
                     metric="Mpixels/sec (Harris+Canny) at 8K frames", batch=4),
}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region."""

    def __init__(self, index):
        self.rows, self.times, self.proc, self.index = [], [], None, index

    def start(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])
            self.times.append(time.perf_counter())

    def count_since(self, t0):
        return sum(1 for t in self.times if t >= t0)

    def stop(self, t0=None, t1=None):
        """Median SM clock / throttle reasons of the samples taken in [t0, t1] (all samples if None)."""
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        rows = [r for r, t in zip(self.rows, self.times) if (t0 is None or t >= t0) and (t1 is None or t <= t1)]
        sm = [float(r[0]) for r in rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 2 + i and r[2 + i].lower().startswith("active") for r in rows)]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm)}


DUMP_SAMPLE = 4 << 20      # elements kept of a larger output by --dump-outputs: <= 48 MB in all for every workload


def dump_outputs(outdir, outputs):
    """Writes {name: array} as outdir/<name>.npy in float32 (float32 and 8/16-bit integer outputs) or float64 (the
    others): exact either way.  An array of more than DUMP_SAMPLE elements is replaced by a fixed seeded sample of its
    rows (of its elements when 1-D), in their original order, so that two builds can be compared entry by entry."""
    os.makedirs(outdir, exist_ok=True)
    for name, a in outputs.items():
        a = np.asarray(a)
        small = a.dtype == np.float32 or (a.dtype.kind in "iub" and a.dtype.itemsize <= 2)
        a = a.astype(np.float32 if small else np.float64)
        row = int(np.prod(a.shape[1:])) if a.ndim > 1 else 1
        if a.size > DUMP_SAMPLE:
            keep = np.sort(np.random.default_rng(0).choice(len(a), DUMP_SAMPLE // row, replace=False, shuffle=False))
            a = a[keep]
        np.save(os.path.join(outdir, name + ".npy"), a)


def grey_of(rgb):
    """dlib's grey rule (r+g+b)/3, pixel.h:775-783."""
    return (rgb.astype(np.uint16).sum(axis=-1) // 3).astype(np.uint8)


def frames_for(workload, seed0, n, distinct):
    """Synthetic frames of a workload (SURVEY.md 8d recipes).  Returns a dict of uint8 arrays."""
    from image_b200 import synth
    w = WORKLOADS[workload]
    nx, ny = w["nx"], w["ny"]
    if workload == "composite":
        rgb = synth.batch(synth.frame_rgb, seed0, n, ny, nx, distinct=min(n, distinct))
        return {"rgb": rgb, "grey": grey_of(rgb)}
    if workload == "surf":
        return {"rgb": synth.batch(synth.frame_blobs, seed0 + 1000, n, ny, nx, distinct=min(n, distinct))}
    return {"grey": synth.batch(synth.frame_shapes, seed0 + 2000, n, ny, nx, distinct=min(n, distinct))}


# ------------------------------------------------------------------------------------------ reference arm
def _cpu_model():
    try:
        for line in open("/proc/cpuinfo"):
            if line.lower().startswith("model name"):
                return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def _host_memory_available():
    """Bytes this process may still allocate: MemAvailable, capped by the cgroup limit when there is one."""
    avail = None
    try:
        for line in open("/proc/meminfo"):
            if line.startswith("MemAvailable:"):
                avail = int(line.split()[1]) * 1024
    except OSError:
        pass
    try:
        mx = open("/sys/fs/cgroup/memory.max").read().strip()
        if mx != "max":
            cur = int(open("/sys/fs/cgroup/memory.current").read())
            avail = min(avail, int(mx) - cur) if avail is not None else int(mx) - cur
    except (OSError, ValueError):
        pass
    return avail


def run_reference(args):
    """The reference's own CPU implementation (oracle/_ref when built, else the oracle port) on the box's host cores, with
    every core busy: a step is `nf` independent frames whose detector calls all go through one thread pool.  Canny, FHOG
    and SURF are single-threaded in the reference; Harris is OpenMP-parallel inside a frame and gets cores/nf threads."""
    from concurrent.futures import ThreadPoolExecutor
    w = WORKLOADS[args.workload]
    nx, ny, dets = w["nx"], w["ny"], w["dets"]
    cores = os.cpu_count() or 1
    mem = _host_memory_available()
    per_frame_gb = 3 if args.workload != "stream8k" else 12     # ~1 GB per 4K Canny call, 0.5 GB Harris
    nf_mem = max(1, int(mem // (per_frame_gb << 30))) if mem else 16
    # a pooled 4K frame costs about 0.5 s of wall time on a 128-core box: keep the whole run near three minutes
    cost = 1.0 if args.workload == "composite" else (1.2 if args.workload == "surf" else 6.0)
    nf_time = max(2, int(360 / cost / (args.steps + min(args.warmup, 1))))
    nf = max(1, args.ref_frames if args.ref_frames > 0 else min(cores, 64, nf_mem, nf_time))
    omp = max(1, cores // nf)
    os.environ["OMP_NUM_THREADS"] = str(omp)                       # read by libgomp when libref_harris.so is loaded below
    from oracle import pyoracle as po
    if po.lib("oracle") is None:
        po.build(ref=False)
        po._cache.clear()
    kind = "reference" if all(po.have_ref(x) for x in ("harris", "canny", "dlib")) else "port"
    impl = "ref" if kind == "reference" else "oracle"
    fr = frames_for(args.workload, 2000, min(nf, 8), 8)
    pick = lambda key, i: fr[key][i % len(fr[key])]                # noqa: E731

    def step():
        with ThreadPoolExecutor(max_workers=cores) as ex:
            jobs = []
            if "canny" in dets:                                    # longest jobs first
                jobs += [ex.submit(po.canny, pick("grey", i), impl=impl, **CANNY_KW) for i in range(nf)]
            if "surf" in dets:
                jobs += [ex.submit(po.surf, pick("rgb", i), SURF_KW["max_points"], SURF_KW["detection_threshold"], impl=impl) for i in range(nf)]
            if "harris" in dets:
                jobs += [ex.submit(po.harris_detect, pick("grey", i), precision=0, impl=impl, **HARRIS_KW) for i in range(nf)]
            if "fhog" in dets:
                jobs += [ex.submit(po.fhog, pick("rgb", i), impl=impl, **FHOG_KW) for i in range(nf)]
            for j in jobs:
                j.result()

    for _ in range(args.warmup if args.warmup < 2 else 1):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = (time.perf_counter() - t0) / args.steps
    mpix = nf * nx * ny / dt / 1e6
    line = {
        "impl": "reference", "metric": w["metric"], "value": mpix, "unit": "Mpixels/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64/f32 (CPU reference)",
        "data": "synthetic",
        "config": {"workload": w["name"], "frames_per_step": nf, "detectors": dets},
        "cpu_baseline": {"value": mpix, "unit": "Mpixels/s", "cores": cores, "cpu_model": _cpu_model(), "omp_num_threads": omp, "kind": kind,
                         "sample": "%d synthetic frame(s) per step (%d distinct), %d steps; all calls of a step in one %d-thread pool, Harris with %d OpenMP thread(s) per frame%s"
                                   % (nf, min(nf, 8), args.steps, cores, omp, "; Canny FFT through the oracle DFT shim (FFTW3 absent)" if kind == "reference" and "canny" in dets else "")},
        "e2e": {"value": mpix, "unit": "Mpixels/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------ GPU arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", default="composite", choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=0, help="frames per GPU per step (0 = the workload's default)")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--ref-frames", type=int, default=0, help="frames per reference step (0 = bounded by cores / memory / time)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--profile-mode", action="store_true", help="device steps only (for ncu launch lists): no per-detector, e2e or CPU legs")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed (rank 0) as DIR/<name>.npy, float32/float64: Harris corner "
                         "counts, raster indices y*nx+x and strengths; Canny edge maps and edge-pixel counts; FHOG features; "
                         "SURF counts and point records; large arrays as a seeded sample (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    wl = WORKLOADS[args.workload]
    NX, NY, dets = wl["nx"], wl["ny"], wl["dets"]

    if args.impl == "reference":
        if rank == 0:
            run_reference(args)
        return

    import torch
    import torch.distributed as dist
    from image_b200 import _lib
    from image_b200 import harris as H
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the product path has no CPU fallback "
                         "(use --impl reference for the CPU reference arm)")
    torch.cuda.set_device(local)
    if world > 1:
        import datetime
        # (a rank that dies must not leave the others waiting for the default ten minutes)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local), timeout=datetime.timedelta(seconds=180))
    lib = _lib.load()
    ctx = _lib.context(local)
    B = args.batch or wl["batch"]
    W = max(args.warmup, 3)
    K = args.steps

    # ---- one process per GPU: stay on the GPU's NUMA node, so that the pinned frame buffers are local to it
    from image_b200.shard import bind_to_gpu_numa
    aff_prev, aff_new = bind_to_gpu_numa(local) if not os.environ.get("B2F_NO_NUMA_BIND") else (os.sched_getaffinity(0), None)

    # ---- synthetic frames (seeded per rank: frames are independent units, sharded across ranks), 8 distinct per rank
    fr = frames_for(args.workload, 2000 + 1000 * rank, B, 8)
    host = {k: torch.from_numpy(v).pin_memory() for k, v in fr.items()}
    dev = {k: v.cuda() for k, v in host.items()}
    in_bytes = sum(v.nbytes for v in fr.values())
    stream = torch.cuda.Stream()          # a real (non-default) stream: the C ABI launches on it and
    torch.cuda.set_stream(stream)         # the CUDA events below are recorded on the same stream
    sp = stream.cuda_stream

    # ---- device-resident outputs, contexts and streams: independent detectors get their own context (stream + scratch)
    cap = 65536
    if "harris" in dets:
        d_R = torch.empty((B, NY, NX), dtype=torch.float32, device="cuda")
        d_xy = torch.empty((B, cap), dtype=torch.int32, device="cuda")
        d_st = torch.empty((B, cap), dtype=torch.float32, device="cuda")
        d_cnt = torch.empty(B, dtype=torch.int32, device="cuda")
    if "canny" in dets:
        from image_b200 import canny as Cn
        d_edges = torch.empty((B, NY, NX), dtype=torch.uint8, device="cuda")
        d_nz = torch.empty(B, dtype=torch.int32, device="cuda")
        ctx_c, st_c, ev_c = _lib.new_context(local), torch.cuda.Stream(), torch.cuda.Event()
    if "fhog" in dets or "surf" in dets:
        from image_b200 import dlib as Dl
    if "fhog" in dets:
        hnr, hnc = Dl.fhog_size(NY, NX, **FHOG_KW)
        d_hog = torch.empty((B, hnr, hnc, 31), dtype=torch.float32, device="cuda")
        ctx_f, st_f, ev_f = _lib.new_context(local), torch.cuda.Stream(), torch.cuda.Event()
    if "surf" in dets:
        surf_rec = torch.empty((B, SURF_KW["max_points"], 70), dtype=torch.float64).pin_memory().numpy()
    ev_fork = torch.cuda.Event()
    ctxs = [ctx] + ([ctx_c] if "canny" in dets else []) + ([ctx_f] if "fhog" in dets else [])
    surf_counts, surf_last = [], {}

    def harris_dev(d_grey):
        # certified path: fused response + error bound -> tolerant NMS -> exact patches -> reference-identical lists
        H.harris_corners_dev(d_grey, True, B, NX, NY, cap, d_xy, d_st, d_cnt, d_R=d_R, stream=sp, **HARRIS_KW)

    def step_dev(frames=None):
        f = frames or dev
        if "surf" in dets:
            _, c = Dl.surf_dev(f["rgb"], B, NY, NX, rec=surf_rec, stream=sp, **SURF_KW)
            surf_counts[:] = [int(c.mean())]
            surf_last["counts"] = c
            return
        ev_fork.record(stream)
        if "canny" in dets:
            st_c.wait_event(ev_fork)
            Cn.canny_dev(f["grey"], B, NX, NY, d_edges, d_nz, stream=st_c.cuda_stream, ctx=ctx_c, **CANNY_KW)
            ev_c.record(st_c)
        if "fhog" in dets:
            st_f.wait_event(ev_fork)
            Dl.fhog_dev(f["rgb"], B, NY, NX, d_hog, stream=st_f.cuda_stream, ctx=ctx_f, **FHOG_KW)
            ev_f.record(st_f)
        harris_dev(f["grey"])
        if "canny" in dets:
            stream.wait_event(ev_c)
        if "fhog" in dets:
            stream.wait_event(ev_f)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, k):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record(stream)
        for _ in range(k):
            fn()
        e1.record(stream)
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device="cuda")
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    def launch_total():
        return sum(int(lib.b2f_launch_count(c)) for c in ctxs)

    # ---- warm-up, then the device-resident timed region (the inputs of a step are far larger than the 126 MB L2,
    #      so every step streams from HBM)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()                      # nvidia-smi needs a moment before its first line: start it before the warm-up
    for _ in range(W):
        step_dev()
    l0 = launch_total()
    t_region0 = time.perf_counter()
    ms_total = timed(step_dev, K)
    t_region1 = time.perf_counter()
    launches = launch_total() - l0
    snap = {}                                # the last timed step's outputs, before anything below overwrites them
    if args.dump_outputs and rank == 0:
        if "surf" in dets:
            snap.update(surf_records=surf_rec.copy(), surf_counts=surf_last["counts"].copy())
        if "harris" in dets:
            snap.update(harris_counts=d_cnt.clone(), harris_xy=d_xy.clone(), harris_strength=d_st.clone())
        if "canny" in dets:
            snap.update(canny_edges=d_edges.clone(), canny_nonzero=d_nz.clone())
        if "fhog" in dets:
            snap.update(fhog=d_hog.clone())
    clocks = None
    if rank == 0:
        note = "timed region"
        if sampler.proc and sampler.count_since(t_region0) < 3 and not args.profile_mode:
            # the timed region is shorter than a few 100 ms sampling periods: keep the very same load running
            # (untimed) until enough samples have arrived, and say so
            t_end = time.perf_counter() + 1.5
            while time.perf_counter() < t_end and sampler.count_since(t_region0) < 4:
                step_dev()
                torch.cuda.synchronize()
            t_region1 = time.perf_counter()
            note = "timed region + untimed continuation of the same steps (region shorter than the 100 ms sampling period)"
        clocks = sampler.stop(t_region0, t_region1)
        clocks["window"] = note
    if snap:
        out = {k: v.cpu().numpy() if torch.is_tensor(v) else v for k, v in snap.items()}
        if "harris_counts" in out:          # the stored part of each frame's corner list, frame after frame
            n = np.minimum(out["harris_counts"], cap)
            for k in ("harris_xy", "harris_strength"):
                out[k] = np.concatenate([out[k][i, :n[i]] for i in range(B)])
        if "surf_counts" in out:
            out["surf_records"] = np.concatenate([out["surf_records"][i, :c] for i, c in enumerate(out["surf_counts"])])
        for k in ("canny_edges", "fhog"):
            if k in out:
                out[k] = out[k].reshape(-1)
        dump_outputs(args.dump_outputs, out)
        del snap, out
    ms_step = ms_total / K
    value = world * B * NX * NY / (ms_step * 1e-3) / 1e6

    if args.profile_mode:
        if rank == 0:
            print(json.dumps({"metric": wl["metric"], "value": value, "unit": "Mpixels/s", "n_gpus": world, "steps": K, "warmup": W,
                              "ms_per_step": ms_step, "profile_mode": True, "gpu_launches": launches, "clocks": clocks}))
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- per-detector device times (explain the headline)
    detail, per_det = {}, {}

    def t_of(fn, k=5):
        fn()                                   # first call may grow the context's scratch arena
        torch.cuda.synchronize()
        return timed(fn, k) / k

    def mpix(ms):
        return B * NX * NY / (ms * 1e-3) / 1e6

    roof = None
    if "harris" in dets:
        th = t_of(lambda: H.harris_response_dev(dev["grey"], True, B, NX, NY, d_R, stream=sp, **HARRIS_KW), 10)
        tall = t_of(lambda: harris_dev(dev["grey"]))
        detail["harris_response_ms"] = th
        detail["harris_certify_nms_ms"] = max(tall - th, 0.0)
        detail["harris_cert_stats_since_start"] = H.cert_stats(ctx)
        per_det["harris"] = {"device_ms_per_frame": tall / B, "device_mpix_s": mpix(tall)}
        # ---- roofline of the dominant target kernel: fused Harris gradient+response, 5 B/px algorithmic
        peak, peak_src = peaks()
        alg_bytes = 5.0 * B * NX * NY
        achieved = alg_bytes / (th * 1e-3) / 1e9
        roof = {"bound": "hbm", "kernel": "harris_fused3_kernel<3,7,64x48 tiles,u8> (one launch: interior and border tiles)",
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "frac_of_nominal_8000": achieved / 8000.0, "traffic": None, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": alg_bytes, "launch_ms": th,
                "note": "this chain is fp32-FMA / shared-memory bound (~137 fp32 lane-ops per 5 algorithmic bytes): "
                        "its HBM fraction cannot exceed ~24 % (DESIGN.md 4.1)"}
        tp = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tp):
            try:
                tj = json.load(open(tp))
                per_px = tj.get("harris_fused3_dram_bytes_per_pixel")
                if per_px:
                    roof["traffic"] = per_px * B * NX * NY
                    roof["traffic_source"] = tj.get("source")
            except Exception:
                pass
    if "canny" in dets:
        detail["canny_ms"] = t_of(lambda: Cn.canny_dev(dev["grey"], B, NX, NY, d_edges, d_nz, stream=sp, **CANNY_KW))
        per_det["canny"] = {"device_ms_per_frame": detail["canny_ms"] / B, "device_mpix_s": mpix(detail["canny_ms"])}
    if "fhog" in dets:
        detail["fhog_ms"] = t_of(lambda: Dl.fhog_dev(dev["rgb"], B, NY, NX, d_hog, stream=sp, **FHOG_KW))
        per_det["fhog"] = {"device_ms_per_frame": detail["fhog_ms"] / B, "device_mpix_s": mpix(detail["fhog_ms"])}
    if "surf" in dets:
        peak, peak_src = peaks()
        alg_bytes = 11.0 * B * NX * NY                 # SURVEY.md 8d: 3 B/px in + int32 SAT written 4 + read once 4
        achieved = alg_bytes / (ms_step * 1e-3) / 1e9
        roof = {"bound": "hbm", "kernel": "SURF pipeline (SAT, Hessian pyramid, 3x3x3 NMS, descriptors) incl. its host sort / filter tail",
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": None, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": alg_bytes, "launch_ms": ms_step,
                "note": "whole step, not one kernel: the fp64 pyramid (132 MB per frame) is materialised and the key-point tail runs on the host"}
        per_det["surf"] = {"device_input_ms_per_frame": ms_step / B, "points_per_frame": surf_counts[0] if surf_counts else None, **SURF_KW}

    # ---- sensitivity: the same step on structure-rich frames (the C2 rectangles + discs recipe at this size: thousands of
    #      corners and long edge chains per frame instead of ~60 corners) — NMS vote-outs, certification, hysteresis and the
    #      Canny fp64 fallback are content dependent
    def timed_local(fn, k):                   # this rank only: no collective inside (used where ranks may diverge)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record(stream)
        for _ in range(k):
            fn()
        e1.record(stream)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)

    sens = None
    if args.workload == "composite" and rank == 0:
        try:
            from image_b200 import synth
            g = synth.batch(synth.frame_shapes, 7000, B, NY, NX, distinct=min(B, 8))
            rich = {"grey": torch.from_numpy(g).cuda(), "rgb": torch.from_numpy(np.repeat(g[..., None], 3, axis=3)).cuda()}
            step_dev(rich)
            torch.cuda.synchronize()
            ks = max(3, K // 2)
            ms = timed_local(lambda: step_dev(rich), ks) / ks
            sens = {"frames": "rectangles + discs + noise (SURVEY.md 8d C2 recipe) at %dx%d, grey replicated to RGB" % (NX, NY),
                    "value": mpix(ms), "unit": "Mpixels/s", "ms_per_step": ms, "scope": "rank 0's GPU only",
                    "corners_per_frame": float(d_cnt.float().mean()), "edge_pixel_fraction": float(d_nz.float().mean()) / (NX * NY)}
            del rich
        except Exception as ex:
            sens = {"error": str(ex)}

    # ---- end to end through the public host API (pinned host in, results back on the host)
    e2e = None
    e2e_error = None
    h2d = d2h = 0
    try:
        from image_b200.features import features_batch
        pin_edges = torch.empty((B, NY, NX), dtype=torch.uint8).pin_memory().numpy() if "canny" in dets else None
        pin_hog = torch.empty((B, hnr, hnc, 31), dtype=torch.float32).pin_memory().numpy() if "fhog" in dets else None
        np_host = {k: v.numpy() for k, v in host.items()}

        def step_e2e():
            nonlocal h2d, d2h
            if "surf" in dets:
                _, c = Dl.surf_batch(np_host["rgb"], raw=True, rec=surf_rec, ctx=ctx, **SURF_KW)
                h2d = np_host["rgb"].nbytes
                d2h = int(c.sum()) * 70 * 8 + 4 * B
                return
            # ONE upload per frame: the RGB frames (composite; grey derived on the device) or the grey stream (stream8k)
            src = np_host["rgb"] if "fhog" in dets else np_host["grey"]
            o = features_batch(src, harris=dict(HARRIS_KW), canny=dict(CANNY_KW), fhog=dict(FHOG_KW) if "fhog" in dets else None,
                               corner_cap=cap, out_edges=pin_edges, out_hog=pin_hog, ctx=ctx)
            h2d = src.nbytes
            d2h = int(o["corners"][3].sum()) * 8 + 8 * B + pin_edges.nbytes + (pin_hog.nbytes if pin_hog is not None else 0)
        for _ in range(2):
            step_e2e()
        e2e_ready = True
    except Exception as ex:   # keep the device-timed line even if the host path fails
        e2e_ready = False
        e2e_error = str(ex)
    # collectives stay outside the try blocks: a rank that failed still takes part in them
    barrier()
    ke = max(2, K // 2)
    dt_local = float("inf")
    if e2e_ready:
        try:
            t0 = time.perf_counter()
            for _ in range(ke):
                step_e2e()
            torch.cuda.synchronize()
            dt_local = (time.perf_counter() - t0) / ke
        except Exception as ex:
            e2e_error = str(ex)
    dt = torch.tensor([dt_local], device="cuda")
    if world > 1:
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
    if np.isfinite(float(dt.item())):
        api = "surf_batch (b2f_surf_batch)" if "surf" in dets else \
              ("features_batch (b2f_features_batch_rgb: one upload of the RGB frames, grey derived on the device; chunked; detectors side by side, copies on their own streams)" if "fhog" in dets
               else "features_batch (b2f_features_batch_grey: one upload of the grey frames; chunked; detectors side by side, copies on their own streams)")
        e2e = {"value": world * B * NX * NY / float(dt.item()) / 1e6, "unit": "Mpixels/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
               "api": api + ", pinned host buffers"}
    else:
        e2e = {"value": None, "unit": "Mpixels/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0, "error": e2e_error if not e2e_ready or dt_local == float("inf") else "another rank failed"}

    # ---- CPU baseline (rank 0, N=1 only): the reference's own code on a bounded sample, in a child process so that its
    #      OpenMP team size and memory stay its own
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            os.sched_setaffinity(0, aff_prev)      # the CPU reference gets every core of the box
            nfr = max(2, min((os.cpu_count() or 2) // 4, 32)) if args.workload != "stream8k" else 4
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--workload", args.workload, "--steps", "1",
                                "--warmup", "0", "--ref-frames", str(nfr)], capture_output=True, text=True, timeout=900)
            pl = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])
            cpu = pl["cpu_baseline"]
        except Exception as ex:
            cpu = {"value": None, "unit": "Mpixels/s", "cores": os.cpu_count(), "kind": "port", "sample": "failed: %s" % ex}

    if rank == 0:
        line = {
            "metric": wl["metric"], "value": value, "unit": "Mpixels/s",
            "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None,
            "dtype": "f64 (SURF)" if "surf" in dets else ("f32 (Harris, FHOG) / f64 (Canny, Harris certification)"), "data": "synthetic",
            "config": {"workload": wl["name"], "detectors": dets, "frames_per_gpu": B, "distinct_frames_per_gpu": min(B, 8),
                       "l2": "inputs larger than L2 (%.0f MB per step)" % (in_bytes / 1e6),
                       "harris_path": "default (certified: lists and strengths bit-identical to the reference)" if "harris" in dets else None,
                       "parallelism": "frames sharded over %d GPU(s), no data-path collective" % world,
                       "host_affinity": ("GPU NUMA node, %d cpus" % len(aff_new)) if aff_new else "unchanged (NUMA node of the GPU unknown)"},
            "clocks": clocks, "e2e": e2e, "gpu_launches": launches, "roofline": roof, "cpu_baseline": cpu,
            "detail_ms_per_step": detail, "per_detector": per_det, "sensitivity": sens,
        }
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
