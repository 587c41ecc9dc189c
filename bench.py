#!/usr/bin/env python
"""bench.py -- throughput of the triangulation hot path (BASELINE.json metric: 3D points/s).

Workload (config 4 of BASELINE.json): synthetic 8-camera ring rig, 100 M frames per GPU, 20 % missing
detections, MatrixTriangulator::triangulatePoints (DLT).  One "step" = one pass of the batch kernel
over all frames of this rank.  Frames are independent, so ranks own contiguous frame ranges of the
global index space (weak scaling: per-GPU work fixed) with no data-path collective; `gathered` adds
the final NCCL all-gather of the points the north star names.

  python bench.py [--gpus N --steps K --warmup W] [--impl reference] [--mode matrix|ray] [--precision f64|f32]
                  [--dump-outputs DIR]

Prints ONE JSON line (rank 0).  `--impl reference` times the CPU restatement of the reference
(oracle/, all host threads) on a bounded sample of the same workload.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "3D points/sec (8-cam DLT, 20% missing)"  # --mode ray swaps in the ray solver, named in config.workload
UNIT = "points/s"
N_CAMS = 8


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--frames", type=int, default=100_000_000, help="frames per GPU")
    ap.add_argument("--mode", default="matrix", choices=["matrix", "ray"])
    ap.add_argument("--precision", default="f64", choices=["f64", "f32"])
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the points the last timed step computed (rank 0's frames) to DIR/<name>.npy (see dump_outputs)")
    a = ap.parse_args()
    if a.steps < 1 or a.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if a.dump_outputs and a.impl != "b200":
        ap.error("--dump-outputs writes what the GPU path computed; the reference arm keeps no outputs")
    return a


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "20"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([v.strip() for v in line.split(",")])

    def __exit__(self, *a):
        if self.proc:
            time.sleep(0.15)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm, mx, reasons = [], 0, set()
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = max(mx, float(r[1]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm)}


def bind_to_gpu_numa_node(index):
    """Pin this rank's threads to the CPU cores next to its GPU (NVML's ideal affinity), so that the page-locked
    host buffers it allocates afterwards live on that NUMA node: with 8 ranks streaming 64 B per frame each,
    remote-socket buffers halve the per-GPU PCIe rate."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        n_words = (os.cpu_count() + 63) // 64
        words = pynvml.nvmlDeviceGetCpuAffinity(h, n_words)
        cpus = {64 * w + b for w, word in enumerate(words) for b in range(64) if word >> b & 1}
        cpus &= set(os.sched_getaffinity(0))
        if cpus:
            os.sched_setaffinity(0, cpus)
            return sorted(cpus)[0], len(cpus)
    except Exception:
        pass
    return None


DUMP_SAMPLE = 1 << 21  # frames kept when the whole output is larger than DUMP_BYTES
DUMP_BYTES = 64 << 20


def dump_outputs(path, xyz):
    """Write the [frames, 3] float32 points of one step as path/xyz_f32.npy.  Above DUMP_BYTES, a fixed, seeded sample
    of the frames (the same one on every run with the same --frames), with their indices in path/frame_index.npy
    (float64, exact for any frame count).  The inputs are a pure function of the frame index, so two builds of the
    project can be compared output for output."""
    import numpy as np
    import torch
    os.makedirs(path, exist_ok=True)
    n = xyz.shape[0]
    if n * xyz.element_size() * 3 <= DUMP_BYTES:
        np.save(os.path.join(path, "xyz_f32.npy"), xyz.cpu().numpy())
        return
    idx = np.unique(np.random.default_rng(0).integers(0, n, DUMP_SAMPLE))
    np.save(os.path.join(path, "xyz_f32.npy"), xyz[torch.from_numpy(idx).to(xyz.device)].cpu().numpy())
    np.save(os.path.join(path, "frame_index.npy"), idx.astype(np.float64))


def oracle_cams(cams):
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle_py as O  # cpu_baseline / reference arm only
    return O, [O.make_camera(c.cam_id, c.width, c.height, c.focal, c.position, c.quat) for c in cams]


def cpu_run(O, ocams, host_xy, mode, threads):
    t0 = time.perf_counter()
    r = O.triangulate_points(ocams, host_xy, O.MATRIX if mode == "matrix" else O.RAY, allow_too_few=True, nthreads=threads)
    dt = time.perf_counter() - t0
    import numpy as np
    valid = int((np.unpackbits(r["mask"].view(np.uint8)).reshape(-1, 32).sum(1) >= 2).sum())
    return valid, dt


def ref_available():
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import ref_py as R  # cpu_baseline / reference arm only
    return R if R.available() else None


def ref_run(R, cams, host_xy, mode, threads):
    """The REFERENCE'S OWN triangulatePoints (oracle/_ref: its sources compiled unmodified against oracle/shim) over the
    frames of host_xy [cams][frames][2] that have >= 2 views (the reference throws on the others,
    MatrixTriangulator.cpp:92-94).  The reference is single-threaded; `threads` independent instances each take a
    contiguous slice of the frames (ctypes releases the GIL).  -> (points, seconds)."""
    import numpy as np
    from concurrent.futures import ThreadPoolExecutor
    xy = np.ascontiguousarray(host_xy, np.float64)
    ok = ((xy[:, :, 0] != -1) & (xy[:, :, 1] != -1)).sum(0) >= 2
    xy = np.ascontiguousarray(xy[:, ok])
    n = xy.shape[1]
    tup = [(c.cam_id, c.width, c.height, c.focal, c.position, c.quat) for c in cams]
    refs = [R.Reference(cams=tup, mode=R.MATRIX if mode == "matrix" else R.RAY) for _ in range(threads)]
    cuts = [n * i // threads for i in range(threads + 1)]
    parts = [np.ascontiguousarray(xy[:, cuts[i]:cuts[i + 1]]) for i in range(threads)]
    t0 = time.perf_counter()
    with ThreadPoolExecutor(threads) as ex:
        list(ex.map(lambda i: refs[i].triangulate_points(parts[i]) if parts[i].shape[1] else None, range(threads)))
    return n, time.perf_counter() - t0


def cpu_baseline(cams, mode, seconds, make_sample):
    """The reference's CPU path on all host cores, on a bounded sample of the same workload: oracle/_ref (the
    reference's own code, "reference") when it was built, else the oracle port ("port")."""
    O, ocams = oracle_cams(cams)
    threads = os.cpu_count() or 1
    n = 200_000
    xy = make_sample(n)
    valid, dt = cpu_run(O, ocams, xy, mode, threads)
    rate = valid / dt
    n2 = int(min(max(rate * seconds, n), 40_000_000))
    xy = make_sample(n2)
    valid, dt = cpu_run(O, ocams, xy, mode, threads)
    v1, dt1 = cpu_run(O, ocams, xy[:, :min(n2, 2_000_000)], mode, 1)  # the reference itself is single-threaded (SURVEY 8b)
    port = {"value": valid / dt, "unit": UNIT, "cores": threads, "kind": "port",
            "sample": "first %d frames of the workload, %d valid points, %.2f s, OpenMP over frames" % (n2, valid, dt),
            "single_thread": v1 / dt1}
    R = ref_available()
    if R is None:
        return port
    m = 100_000
    pts, dt = ref_run(R, cams, xy[:, :m], mode, threads)
    m2 = int(min(max(pts / dt * seconds, m), n2))
    pts, dt = ref_run(R, cams, xy[:, :m2], mode, threads)
    p1, d1 = ref_run(R, cams, xy[:, :min(m2, 200_000)], mode, 1)
    return {"value": pts / dt, "unit": UNIT, "cores": threads, "kind": "reference",
            "sample": "the %d frames with >= 2 views among the first %d of the workload, %.2f s, %d independent instances of the "
                      "reference's MatrixTriangulator::triangulatePoints (oracle/_ref), one per host thread" % (pts, m2, dt, threads),
            "single_thread": p1 / d1, "port": port}


def reference_arm(a, emit):
    """--impl reference: the reference's CPU implementation of the path on this box -- oracle/_ref (the reference's own
    sources, compiled unmodified against oracle/shim; one single-threaded instance per host core) when it was built,
    else the oracle port (OpenMP over frames)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import tri_b200 as T  # host-side camera arithmetic + synthetic generator only
    from tri_b200 import synthetic as S
    cams = S.ring_rig(N_CAMS)
    O, ocams = oracle_cams(cams)
    R = ref_available()
    threads = os.cpu_count() or 1
    kind = "reference" if R is not None else "port"

    def run(xy):
        return ref_run(R, cams, xy, a.mode, threads) if R is not None else cpu_run(O, ocams, xy, a.mode, threads)
    probe = S.generate_frames(cams, 200_000).numpy()
    valid, dt = run(probe)
    per_step_s = min(20.0, 150.0 / max(a.steps + a.warmup, 1))
    n = int(min(max(valid / dt * per_step_s, 200_000), 40_000_000))
    xy = S.generate_frames(cams, n).numpy()
    for _ in range(a.warmup):
        run(xy)
    tot_valid, tot_t = 0, 0.0
    for _ in range(a.steps):
        v, dt = run(xy)
        tot_valid += v
        tot_t += dt
    val = tot_valid / tot_t
    sample = ("%d frames per step (first frames of the workload), " % n) + (
        "%d independent single-threaded instances of the reference's triangulatePoints (oracle/_ref)" % threads if R is not None
        else "oracle port, OpenMP over frames")
    emit({
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps,
        "warmup": a.warmup, "ms_per_step": 1e3 * tot_t / a.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "synthetic 8-camera ring rig, 20%% missing detections, DLT (%s); CPU sample %s" % (a.mode, sample)},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": threads, "kind": kind, "sample": sample},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0})


def main():
    a = parse()
    # stdout carries exactly ONE JSON line: anything a library prints there meanwhile (NCCL's version banner does)
    # is sent to stderr; the real stdout comes back for the final print.
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    def emit(obj):
        sys.stdout.flush()
        os.dup2(real_stdout, 1)
        print(json.dumps(obj), flush=True)

    if a.impl == "reference":
        return reference_arm(a, emit)
    import torch
    import torch.distributed as dist
    import tri_b200 as T
    from tri_b200 import synthetic as S

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the engine has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    all_cpus = os.sched_getaffinity(0)
    numa = bind_to_gpu_numa_node(local)  # the pinned host buffers of the e2e leg are first-touched after this
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    cams = S.ring_rig(N_CAMS)
    eng = T.Engine(cams, local)
    F = a.frames
    from tri_b200 import sharding as SH
    frame0, frame1 = SH.shard_range(world * F, rank, world)  # contiguous range of the global frame index space
    assert frame1 - frame0 == F
    mode = T.MATRIX if a.mode == "matrix" else T.RAY
    flags = T.ALLOW_TOO_FEW | (T.F32 if a.precision == "f32" else 0)
    xy = S.generate_frames(cams, F, frame0=frame0, device=dev)  # [8, F, 2] float32, resident in HBM
    out = {"xyz_f32": torch.empty((F, 3), dtype=torch.float32, device=dev)}
    algo_bytes = (8 * N_CAMS + 12) * F

    def step(fl=flags, o=out):
        eng.triangulate_points_device(mode, xy, fl, out=o)

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        barrier()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
        l0 = eng.kernel_launches
        ev[0].record()
        for i in range(steps):
            fn()
            ev[i + 1].record()
        barrier()
        total = ev[0].elapsed_time(ev[-1])
        per = [ev[i].elapsed_time(ev[i + 1]) for i in range(steps)]
        t = torch.tensor([total], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), per, eng.kernel_launches - l0

    # valid points per step (frames with >= 2 views), counted once from the masks
    m = eng.triangulate_points_device(mode, xy, flags, want=("xyz_f32", "mask"))
    eng.device_status()
    pop = torch.zeros_like(m["mask"])
    for c in range(N_CAMS):
        pop += (m["mask"] >> c) & 1
    valid = torch.tensor([int((pop >= 2).sum())], dtype=torch.int64, device=dev)
    del m, pop
    if world > 1:
        dist.all_reduce(valid)
    valid_total = int(valid.item())
    torch.cuda.empty_cache()

    clk = ClockSampler(local)
    clk.__enter__()  # sampled over the timed region and the companion kernel timings that follow (all HBM-resident passes)
    total_ms, per, launches = timed(step, a.steps, a.warmup)
    eng.device_status()
    if a.dump_outputs and rank == 0:  # before the companion timings below write other kernels' points into `out`
        dump_outputs(a.dump_outputs, out["xyz_f32"])
    ms_per_step = total_ms / a.steps
    value = valid_total / (ms_per_step * 1e-3)
    kernel_ms = sum(per) / len(per)
    achieved = algo_bytes / (kernel_ms * 1e-3) / 1e9
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    traffic = None
    try:  # per-launch DRAM bytes of this kernel from the committed ncu --set full capture (same 100 M-frame launch)
        t = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json"))).get("%s_%s" % (a.mode, a.precision))
        traffic = float(t) * (F / 100_000_000) if t else None
    except Exception:
        pass
    kname = {("matrix", "f64"): "stream_kernel<DltTile64<MASK_SELECT_HI>, 8 cams, float2, 2-stage ring, 2 CTAs/SM>",
             ("matrix", "f32"): "stream_kernel<DltX2Tile (FFMA2), 8 cams, float2, 2-stage ring, 3 CTAs/SM>",
             ("ray", "f64"): "stream_kernel<RayTableTile<double, closed form>, 8 cams>", ("ray", "f32"): "stream_kernel<RayX2Tile (FFMA2)>"}
    roof = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "frac_of_nominal_8tbs": achieved / 8000.0,
            "traffic": traffic, "algorithmic_bytes_per_launch": algo_bytes, "peak_source": "measured (MEASURED_PEAKS.json)" if peaks else "fallback 6.65 TB/s",
            "kernel": kname[(a.mode, a.precision)],
            "algorithmic_bytes_per_frame": 8 * N_CAMS + 12, "kernel_ms": kernel_ms}

    if a.precision == "f64" and a.mode == "matrix":
        # secondary roofline: the FP64 pipe.  Peak = measured DFMA issue rate (tools/micro/fma_rate.cu: 1.94 warp-inst/clk/SM
        # = 62 lanes) x 148 SMs x 1965 MHz x 2; flops per frame = 56 * C_valid + 80 (SURVEY 8d), C_valid = 6.4 for p_missing = 0.2.
        dfma_peak = 1.94 * 32 * 148 * 1.965e9 * 2 / 1e12
        fl = (56 * 6.4 + 80) * F / (kernel_ms * 1e-3) / 1e12
        roof["fp64_pipe"] = {"achieved_tflops": fl, "peak_tflops": dfma_peak, "frac": fl / dfma_peak,
                             "executed_frac": (56 * 8 + 80) * F / (kernel_ms * 1e-3) / 1e12 / dfma_peak,
                             "note": "absent views still issue (masked), so the pipe executes 56*8+80 flops per frame; a DFMA costs the FP64 "
                                     "pipe one cycle per distinct register-pair source (three-source DFMAs issue at 2/3 rate, "
                                     "tools/micro/dfma_rf.cu): 1164 pipe cycles per pair of frames, 84 % busy (DESIGN.md 3)"}
    res = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
           "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
           "dtype": a.precision, "data": "synthetic",
           "config": {"workload": "synthetic 8-camera ring rig, %d frames per GPU, 20%% missing detections, %s" %
                      (F, "MatrixTriangulator DLT" if a.mode == "matrix" else "RayTriangulator (closed-form minimiser)"),
                      "frames_per_gpu": F, "cameras": N_CAMS, "valid_points_per_step": valid_total,
                      "l2": "inputs (%.1f GB) and outputs (%.1f GB) per step exceed the 126 MB L2; no flush needed" %
                      (8 * N_CAMS * F / 1e9, 12 * F / 1e9), "sharding": "contiguous frame ranges, no data-path collective"},
           "roofline": roof, "gpu_launches": launches}

    # strong scaling beside the weak headline: BASELINE config 4 is "100 M frames at 1/2/4/8 B200" -- the same kernel on
    # this rank's 1/N cut of ONE 100 M-frame batch (launch, tail and skew effects that weak scaling hides show here)
    if world > 1:
        s0, s1 = SH.shard_range(F, rank, world)
        xs = xy[:, s0:s1]
        outs = {"xyz_f32": out["xyz_f32"][:s1 - s0]}

        def step_strong():
            eng.triangulate_points_device(mode, xs, flags, out=outs)
        tms, _, _ = timed(step_strong, a.steps, a.warmup)
        res["strong"] = {"scaling": "strong", "frames_total": F, "frames_per_gpu": s1 - s0, "ms_per_step": tms / a.steps,
                         "value": valid_total / world / (tms / a.steps * 1e-3), "unit": UNIT,
                         "note": "value = valid points of the 100 M-frame batch / max-over-ranks time of one pass over each rank's cut"}

    # the other arithmetic precision and the ray kernel on the same frames, for context
    other = {}
    for name, md, fl in (("dlt_f32" if a.precision == "f64" else "dlt_f64", T.MATRIX, flags ^ T.F32),
                         ("ray_lm_f64", T.RAY, T.ALLOW_TOO_FEW | T.RAY_ANALYTIC_LM), ("ray_closed_f64", T.RAY, T.ALLOW_TOO_FEW),
                         ("ray_closed_f32", T.RAY, T.ALLOW_TOO_FEW | T.F32)):
        def fn(md=md, fl=fl):
            eng.triangulate_points_device(md, xy, fl, out=out)
        tms, _, _ = timed(fn, max(3, a.steps // 2), 2)
        k = tms / max(3, a.steps // 2)
        other[name] = {"ms_per_step": k, "value": valid_total / (k * 1e-3), "hbm_gbs": algo_bytes / (k * 1e-3) / 1e9,
                       "frac": algo_bytes / (k * 1e-3) / 1e9 / peak}
        eng.device_status()
    res["other_kernels"] = other

    # BASELINE config 5's batch half: the 32-camera two-ring rig, ray-LM and DLT on 20 M frames per GPU (the classifier
    # half of that config is exponential in the camera count and not runnable with reference semantics, DESIGN.md 1)
    try:
        F32C = max(512, min(20_000_000, F // 5))
        cams32 = S.ring_rig(32, rings=((6000.0, 3000.0), (9000.0, 5000.0)))
        eng32 = T.Engine(cams32, local)
        xy32 = S.generate_frames(cams32, F32C, frame0=frame0, device=dev)
        out32 = {"xyz_f32": torch.empty((F32C, 3), dtype=torch.float32, device=dev)}
        bytes32 = (8 * 32 + 12) * F32C
        c5 = {"cameras": 32, "frames_per_gpu": F32C, "algorithmic_bytes_per_frame": 8 * 32 + 12}
        for name, md, fl in (("ray_lm_f64", T.RAY, T.ALLOW_TOO_FEW | T.RAY_ANALYTIC_LM), ("ray_closed_f64", T.RAY, T.ALLOW_TOO_FEW),
                             ("ray_closed_f32", T.RAY, T.ALLOW_TOO_FEW | T.F32),
                             ("dlt_f64", T.MATRIX, T.ALLOW_TOO_FEW), ("dlt_f32", T.MATRIX, T.ALLOW_TOO_FEW | T.F32)):
            def fn32(md=md, fl=fl):
                eng32.triangulate_points_device(md, xy32, fl, out=out32)
            tms, _, _ = timed(fn32, 3, 2)
            k = tms / 3
            c5[name] = {"ms_per_step": k, "frames_per_s": world * F32C / (k * 1e-3), "hbm_gbs": bytes32 / (k * 1e-3) / 1e9,
                        "frac": bytes32 / (k * 1e-3) / 1e9 / peak}
            eng32.device_status()
        res["config5_batch_32cam"] = c5
        del xy32, out32, eng32
        torch.cuda.empty_cache()
    except Exception as exc:  # noqa: BLE001
        res["config5_batch_32cam"] = {"error": repr(exc)}

    # BASELINE config 3 (S09_D6, 8 cameras, 6 drones, 3000 frames): the batched DroneClassifier through tri_classify,
    # wall clock of the whole call from host CSR detections to host paths (the fixture ships with the tests)
    if rank == 0:
        try:
            import numpy as np
            gdir = os.path.join(ROOT, "tests", "golden")
            z = np.load(os.path.join(gdir, "S09_D6_dets.npz"))
            ceng = T.Engine(T.load_cameras_xml(os.path.join(gdir, "S09_D6_cameras.xml")), local)
            counts = z["counts"].astype(np.int64)  # [cam][frame] detection counts -> CSR offsets, cameras back to back
            c_nf = counts.shape[1]
            c_offs = np.zeros((counts.shape[0], c_nf + 1), np.int64)
            c_offs[:, 1:] = np.cumsum(counts, axis=1)
            c_offs += np.concatenate([[0], np.cumsum(counts.sum(1))[:-1]])[:, None]
            c_offs, c_xy = c_offs.astype(np.int32).reshape(-1), z["xy"].astype(np.float64)
            ceng.classify(T.MATRIX, 6, c_offs, c_xy, c_nf)
            t0 = time.perf_counter()
            cr = ceng.classify(T.MATRIX, 6, c_offs, c_xy, c_nf)
            cdt = time.perf_counter() - t0
            res["config3_classifier"] = {"dataset": "S09_D6", "mode": "matrix", "n_drones": 6, "frames": c_nf, "seconds": cdt,
                                         "frames_per_s": c_nf / cdt, "candidate_solves": cr["stats"]["solves"],
                                         "points": int(cr["stats"]["phase1"] + cr["stats"]["phase2"]),
                                         "enumerate_ms": cr["stats"]["enumerate_us"] / 1e3, "link_ms": cr["stats"]["link_us"] / 1e3,
                                         "link_us_per_frame": cr["stats"]["link_us"] / c_nf}
        except Exception as exc:  # noqa: BLE001
            res["config3_classifier"] = {"error": repr(exc)}

    # BASELINE config 5's classifier half at the camera count the reference's semantics can run (8; SURVEY F4): 6 simulated
    # drones, detections in permuted order, 20 % dropped (synthetic.generate_multi_drone).  (a) ONE sequence: linking is
    # sequential in the frames (DroneClassifier.cpp:112-144), so this is the latency-bound number; (b) 1 M frames as 1000
    # recordings of 1000 frames through tri_classify_sequences: every recording links on its own CTA.
    if rank == 0:
        try:
            import numpy as np
            cams8 = S.ring_rig(8)
            ceng8 = T.Engine(cams8, local)
            n_one, n_seq, seq_len = 100_000, 1000, 1000
            offs5, xy5, _ = S.generate_multi_drone(cams8, n_seq * seq_len, 6, device=dev)
            from tri_b200 import sharding as SH5
            o1, x1 = SH5.slice_csr(offs5, xy5, 8, n_seq * seq_len, 0, n_one)
            ceng8.classify(T.MATRIX, 6, o1, x1, n_one)  # warm-up (allocations)
            t0 = time.perf_counter()
            r1 = ceng8.classify(T.MATRIX, 6, o1, x1, n_one)
            t_one = time.perf_counter() - t0
            bounds = np.arange(0, n_seq * seq_len + 1, seq_len, dtype=np.int32)
            ceng8.classify_sequences(T.MATRIX, 6, bounds, offs5, xy5, n_seq * seq_len)
            t0 = time.perf_counter()
            rm = ceng8.classify_sequences(T.MATRIX, 6, bounds, offs5, xy5, n_seq * seq_len)
            t_many = time.perf_counter() - t0
            # parity on a sampled sub-sequence: the first 250 frames against the CPU oracle (checker only)
            O5, oc5 = oracle_cams(cams8)
            o2, x2 = SH5.slice_csr(offs5, xy5, 8, n_seq * seq_len, 0, 250)
            ref5 = O5.classify(oc5, O5.MATRIX, 6, o2, x2, 8, 250)
            same = bool(np.array_equal(ref5["assign"], rm["assign"][:, :250]) and np.array_equal(ref5["phase"], rm["phase"][:, :250]))
            res["config5_classifier"] = {
                "cameras": 8, "n_drones": 6, "mode": "matrix",
                "one_sequence": {"frames": n_one, "seconds": t_one, "frames_per_s": n_one / t_one, "points": int(r1["stats"]["phase1"] + r1["stats"]["phase2"]),
                                 "candidate_solves": r1["stats"]["solves"], "enumerate_ms": r1["stats"]["enumerate_us"] / 1e3,
                                 "link_ms": r1["stats"]["link_us"] / 1e3, "link_us_per_frame": r1["stats"]["link_us"] / n_one},
                "many_sequences": {"sequences": n_seq, "frames": n_seq * seq_len, "seconds": t_many, "frames_per_s": n_seq * seq_len / t_many,
                                   "points": int(rm["stats"]["phase1"] + rm["stats"]["phase2"]), "candidate_solves": rm["stats"]["solves"],
                                   "enumerate_ms": rm["stats"]["enumerate_us"] / 1e3, "link_ms": rm["stats"]["link_us"] / 1e3},
                "oracle_parity_first_250_frames": same,
                "cameras_32": None,
                "note": "wall clock of the whole call, host CSR detections in, host paths / assignments out"}
            del offs5, xy5, r1, rm
            # the configuration's own camera count: 32 cameras on two rings.  The enumeration the reference does there is ~6 * 2^26
            # leaves per frame -- not runnable by the reference, the oracle or the enumerating kernels -- so this is the lazy
            # best-first search (tri_classify_lazy.cu), bit-identical to the enumeration at 8 and 12 cameras (tests/).
            cams32 = S.ring_rig(32, rings=((6000.0, 3000.0), (9000.0, 5000.0)))
            ceng32 = T.Engine(cams32, local)
            n32, q32, l32 = 2000, 128, 250
            offs32, xy32, truth32 = S.generate_multi_drone(cams32, q32 * l32, 6, device=dev)
            o3, x3 = SH5.slice_csr(offs32, xy32, 32, q32 * l32, 0, n32)
            ceng32.classify(T.MATRIX, 6, o3, x3, n32)
            t0 = time.perf_counter()
            r3 = ceng32.classify(T.MATRIX, 6, o3, x3, n32)
            t_32 = time.perf_counter() - t0
            b32 = np.arange(0, q32 * l32 + 1, l32, dtype=np.int32)
            t0 = time.perf_counter()
            r4 = ceng32.classify_sequences(T.MATRIX, 6, b32, offs32, xy32, q32 * l32)
            t_32m = time.perf_counter() - t0
            dmin = [float(np.median(np.linalg.norm(r3["paths"][pp][:, None, :] - truth32[:, :n32].transpose(1, 0, 2), axis=2).min(axis=1))) for pp in range(6)]
            res["config5_classifier"]["cameras_32"] = {
                "cameras": 32, "n_drones": 6, "mode": "matrix", "search": "lazy best-first (TRI_CLS_LAZY path, automatic above 16 cameras)",
                "one_sequence": {"frames": n32, "seconds": t_32, "frames_per_s": n32 / t_32, "points": int(r3["stats"]["phase1"] + r3["stats"]["phase2"]),
                                 "nodes_visited": r3["stats"]["nodes"], "solves": r3["stats"]["solves"], "link_us_per_frame": r3["stats"]["link_us"] / n32,
                                 "median_mm_from_simulated_truth_per_path": dmin, "cameras_per_point": float((r3["assign"] > 0).sum(axis=2).mean())},
                "many_sequences": {"sequences": q32, "frames": q32 * l32, "seconds": t_32m, "frames_per_s": q32 * l32 / t_32m,
                                   "points": int(r4["stats"]["phase1"] + r4["stats"]["phase2"])}}
            del offs32, xy32, r3, r4
        except Exception as exc:  # noqa: BLE001
            res.setdefault("config5_classifier", {})["error"] = repr(exc)

    # the frame-sharded classifier (SURVEY 8e): every rank enumerates its frame range of S09_D6 with the trajectory-exact LM,
    # the linking chain hands the tracking state from rank to rank (one point-to-point message each)
    if world > 1:
        try:
            import numpy as np
            gdir = os.path.join(ROOT, "tests", "golden")
            z = np.load(os.path.join(gdir, "S09_D6_dets.npz"))
            seng = T.Engine(T.load_cameras_xml(os.path.join(gdir, "S09_D6_cameras.xml")), local)
            counts = z["counts"].astype(np.int64)
            s_nf = counts.shape[1]
            s_offs = np.zeros((counts.shape[0], s_nf + 1), np.int64)
            s_offs[:, 1:] = np.cumsum(counts, axis=1)
            s_offs += np.concatenate([[0], np.cumsum(counts.sum(1))[:-1]])[:, None]
            s_offs, s_xy = s_offs.astype(np.int32).reshape(-1), z["xy"].astype(np.float64)
            for md, fl, name in ((T.RAY, T.RAY_REFERENCE_LM, "ray_reference_lm"), (T.MATRIX, 0, "matrix")):
                SH.classify_sharded(seng, md, 6, s_offs, s_xy, s_nf, rank, world, fl)
                barrier()
                t0 = time.perf_counter()
                rs = SH.classify_sharded(seng, md, 6, s_offs, s_xy, s_nf, rank, world, fl)
                barrier()
                dt_s = time.perf_counter() - t0
                res.setdefault("config3_classifier_sharded", {})[name] = {"frames": s_nf, "seconds": dt_s, "frames_per_s": s_nf / dt_s,
                                                                          "rank0_enumerate_ms": rs["stats"]["enumerate_us"] / 1e3}
        except Exception as exc:  # noqa: BLE001
            res["config3_classifier_sharded"] = {"error": repr(exc)}

    # final gather of the points over NVLink (north star): one all-gather per step
    if world > 1:
        allp = torch.empty((world * F, 3), dtype=torch.float32, device=dev)

        def step_gather():
            step()
            dist.all_gather_into_tensor(allp, out["xyz_f32"])
        tms, _, _ = timed(step_gather, a.steps, 2)
        res["gathered"] = {"ms_per_step": tms / a.steps, "value": valid_total / (tms / a.steps * 1e-3), "unit": UNIT,
                           "collective": "ncclAllGather of float3 points, %.2f GB per rank" % (12 * F / 1e9)}
        # the same gather FUSED into the kernel: every rank's epilogue stores its points straight into rank 0's
        # result array over NVLink (CUDA-IPC alias of the root buffer), no collective on the data path
        try:
            root_ptr = SH.open_root_buffer(eng, world * F * 12, rank, world)
            stream = torch.cuda.current_stream(dev).cuda_stream
            stride = xy.stride(0) // 2

            def step_fused():
                eng.triangulate_points_device_raw(mode, flags, xy.data_ptr(), N_CAMS, F, stride, root_ptr + rank * F * 12, stream)
            tms, _, _ = timed(step_fused, a.steps, 2)
            ok = True
            if rank == 0:  # the root's array now holds every rank's points, in global frame order
                chk = torch.empty((world * F, 3), dtype=torch.float32, device=dev)
                eng.copy_device(chk.data_ptr(), root_ptr, world * F * 12)
                ok = bool(torch.equal(chk, allp))
                del chk
            res["gathered_fused"] = {"ms_per_step": tms / a.steps, "value": valid_total / (tms / a.steps * 1e-3), "unit": UNIT,
                                     "how": "kernel epilogue stores into rank 0's array over NVLink (CUDA IPC peer memory), gather to root",
                                     "matches_nccl_gather": ok}
            barrier()
            SH.close_root_buffer(eng, root_ptr, rank)
        except Exception as ex:  # e.g. no peer access between the GPUs of this box
            res["gathered_fused"] = {"unavailable": str(ex)[:200]}
        del allp
    clk.__exit__()
    res["clocks"] = clk.summary()

    # end to end through the C ABI with HOST buffers: pinned input, chunked H2D / kernel / D2H pipeline
    if not a.no_e2e:
        h_xy = torch.empty((N_CAMS, F, 2), dtype=torch.float32, pin_memory=True)
        h_out = torch.empty((F, 3), dtype=torch.float32, pin_memory=True)
        h_xy.copy_(xy)
        torch.cuda.synchronize()

        def e2e_step():
            eng.triangulate_points_raw(mode, flags, h_xy.data_ptr(), N_CAMS, F, F, xyz_f32_ptr=h_out.data_ptr())
        esteps = max(2, min(a.steps, 5))
        e2e_step()
        barrier()
        l0 = eng.kernel_launches
        t0 = time.perf_counter()
        for _ in range(esteps):
            e2e_step()
        torch.cuda.synchronize()
        t = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e_s = float(t.item()) / esteps
        res["e2e"] = {"value": valid_total / e_s, "unit": UNIT, "h2d_bytes_per_step": 8 * N_CAMS * F,
                      "d2h_bytes_per_step": 12 * F, "ms_per_step": e_s * 1e3, "steps": esteps,
                      "api": "tri_triangulate_points (host buffers, pinned), per rank",
                      "pcie_gbs": (8 * N_CAMS * F + 12 * F) / e_s / 1e9, "kernel_launches": eng.kernel_launches - l0,
                      "cpu_affinity": numa}
        # the ceiling of that path on this box, with all ranks copying at once: the bare pinned copies of one step's bytes,
        # H2D and D2H concurrently on two streams, no kernel
        d_probe = torch.empty_like(xy)
        s_in, s_out = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
        barrier()
        t0 = time.perf_counter()
        for _ in range(2):
            with torch.cuda.stream(s_in):
                d_probe.copy_(h_xy, non_blocking=True)
            with torch.cuda.stream(s_out):
                h_out.copy_(out["xyz_f32"], non_blocking=True)
            s_in.synchronize()
            s_out.synchronize()
        t = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        res["e2e"]["bare_copy_ms_per_step"] = float(t.item()) / 2 * 1e3
        res["e2e"]["bare_copy_gbs_per_gpu"] = (8 * N_CAMS * F + 12 * F) / (float(t.item()) / 2) / 1e9
        res["e2e"]["fraction_of_bare_copy_ceiling"] = res["e2e"]["bare_copy_ms_per_step"] / res["e2e"]["ms_per_step"]
        del d_probe
        e2e_step()  # h_out holds the end-to-end result again (the probe wrote over it)
        step()
        torch.cuda.synchronize()
        same = bool(torch.equal(h_out[:4000000].to(dev), out["xyz_f32"][:4000000]))
        res["e2e"]["matches_device_path"] = same
        # the same call with the compact ushort2 pixel format (integer detections, 4 B instead of 8 B over PCIe)
        h16 = torch.empty((N_CAMS, F, 2), dtype=torch.uint16, pin_memory=True)
        for c in range(N_CAMS):
            v = xy[c]
            h16[c].copy_(torch.where(v < 0, torch.full_like(v, 65535.0), v).to(torch.int32).to(torch.uint16))
        torch.cuda.synchronize()

        def e2e16():
            eng.triangulate_points_raw(mode, flags | T.PIX_U16, h16.data_ptr(), N_CAMS, F, F, xyz_f32_ptr=h_out.data_ptr())
        e2e16()
        barrier()
        t0 = time.perf_counter()
        for _ in range(esteps):
            e2e16()
        torch.cuda.synchronize()
        t = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e16 = float(t.item()) / esteps
        res["e2e_u16"] = {"value": valid_total / e16, "unit": UNIT, "h2d_bytes_per_step": 4 * N_CAMS * F, "d2h_bytes_per_step": 12 * F,
                          "ms_per_step": e16 * 1e3, "matches_device_path": bool(torch.equal(h_out[:4000000].to(dev), out["xyz_f32"][:4000000]))}
        del h_xy, h_out, h16

    os.sched_setaffinity(0, all_cpus)  # the CPU baseline uses every host core again
    if rank == 0 and world == 1 and not a.no_cpu:
        res["cpu_baseline"] = cpu_baseline(cams, a.mode, a.cpu_seconds, lambda n: xy[:, :n].cpu().numpy())
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0:
        emit(res)


if __name__ == "__main__":
    main()
