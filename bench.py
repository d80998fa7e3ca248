#!/usr/bin/env python
"""bench.py -- POIs/sec of the FFT-CC -> IC-GN hot path (BASELINE.json metric) on N B200s.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--config B|C|D|A|E|F] [--impl ours|reference] [--dump-outputs DIR]
  N>1: python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A step = one pass of the hot path (FFT-CC initial guess + IC-GN to convergence, prepare() included)
over one batch of synthetic POIs.  At N=1 the default workload is BASELINE.json configs[1]
("2D DIC 2048x2048 synthetic speckle, 50k POIs, 33x33 subset, FFTCC->ICGN2D1").  For N>1 every rank
works on its own 50k-POI shard of a denser grid on the same image pair (weak scaling; the path shards over
independent POIs, so there is NO data-path collective: every rank moves its own host buffers over its own
PCIe link).

  value  : whole-job POIs/s with images and the pristine POI queue resident in HBM
           (sum over ranks of POIs / max-over-ranks device time, CUDA events, L2 flushed between steps)
  e2e    : same metric through the host-buffer C-ABI calls (pinned host memory), per rank: image H2D,
           prepare, POI H2D, kernels, POI D2H inside the timed region; max over ranks
  e2e_u8_images: the e2e step with the pair handed over as 8-bit arrays (what the image files hold), N=1 only
  e2e_shim: the same step through the C++ shim (examples/shim_bench.cpp: the reference's class API, the caller's pageable
           Image2D / std::vector<POI2D>), rank 0 only, 2D configs
  capi_multi: ONE process driving all N devices through a GROUP context of the C ABI (ocb_create_multi): the weak
           workload as one queue of N x 50k POIs, and BASELINE.json's other configs -- C (2048^2, 50k POIs, ICGN2D2), E (4096^2, 500k POIs)
           and D (256^3, 20k POIs) -- sharded over the N devices (strong scaling), each with host buffers (e2e); rank 0 only, the
           other ranks idle
  cold_start: a fresh process's ocb_create() and first calls (rank 0, N=1 only)
  roofline: dominant kernel (IC-GN) algorithmic bytes / its CUDA-event time vs MEASURED_PEAKS hbm_gbs; `traffic` and
           `binding_resources_ncu` (issue-slot / FMA / shared-memory pipe utilisation) come from the committed ncu capture
  cpu_baseline: the oracle port of the reference (oracle/, g++ -O3 -fopenmp, nproc-1 threads like
           the reference examples) timed on this box's host cores on the same workload

--impl reference times the reference's own CPU implementation of the path (here: the oracle port,
because the reference cannot be compiled without Eigen/FFTW/OpenCV -- DESIGN.md) on the same config.
"""
import argparse
import gc
import json
import math
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "POIs/sec (FFTCC+ICGN to convergence)"
UNIT = "POI/s"

# algorithmic bytes per POI (SURVEY.md section 8(d)): f32 tiles read once + POI record in/out
def icgn_bytes_per_poi(kind, r):
    if kind == "2d":
        return (2 * r + 5) ** 2 * 4 + (2 * r + 4) ** 2 * 4 + 200
    return (2 * r + 5) ** 3 * 4 + (2 * r + 4) ** 3 * 4 + 248


def fftcc_bytes_per_poi(kind, r):
    if kind == "2d":
        return 2 * (2 * r) ** 2 * 4 + 200
    return 2 * (2 * r) ** 3 * 4 + 248


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def make_workload(cfg_name, rank, world, device=None):
    from opencorr_b200 import synth
    cfg = dict(synth.CONFIGS[cfg_name])
    if cfg["kind"] == "2d":
        w, h = cfg["size"]
        ref, tar = synth.speckle_pair_2d(w, h, second_order=(cfg["order"] == 2), device=device)
        x0, y0, nx, ny, sx, sy = cfg["grid"]
        # weak scaling: rank k takes the same grid shifted by k pixels in x (distinct POIs, same count)
        xy = synth.grid_2d(x0 + rank, y0, nx, ny, sx, sy)
        cfg["n_poi"] = xy.shape[0]
        return cfg, ref, tar, xy
    dx, dy, dz = cfg["size"]
    ref, tar = synth.speckle_pair_3d(dx, dy, dz, device=device)
    x0, y0, z0, nx, ny, nz, sx, sy, sz = cfg["grid"]
    xyz = synth.grid_3d(x0 + rank, y0, z0, nx, ny, nz, sx, sy, sz)
    cfg["n_poi"] = xyz.shape[0]
    return cfg, ref, tar, xyz


DUMP_LIMIT_BYTES = 64 * 1000 * 1000


def dump_outputs(out_dir, pois, rank=0, world=1):
    """--dump-outputs: the POI records the timed path returned in its last step, as out_dir/pois.npy (one rank) or
    pois_rank<k>.npy, float32 [n, 25] (POI2D) / [n, 31] (POI3D).  Every record carries its own coordinates, so two runs can be
    matched row for row.  Above this rank's share of DUMP_LIMIT_BYTES a fixed, seeded sample of rows is written, in queue order."""
    os.makedirs(out_dir, exist_ok=True)
    pois = np.ascontiguousarray(pois, dtype=np.float32)
    budget = DUMP_LIMIT_BYTES // world - 4096  # room for the .npy header
    if pois.nbytes > budget:
        keep = budget // (pois.shape[1] * 4)
        pois = pois[np.sort(np.random.default_rng(0).choice(len(pois), keep, replace=False))]
    np.save(os.path.join(out_dir, "pois.npy" if world == 1 else "pois_rank%d.npy" % rank), pois)


def workload_name(cfg_name, cfg):
    if cfg["kind"] == "2d":
        return "%s: 2D DIC %dx%d synthetic speckle, %d POIs, %dx%d subset, FFTCC2D->ICGN2D%d" % (
            cfg_name, cfg["size"][0], cfg["size"][1], cfg["n_poi"], 2 * cfg["r"] + 1, 2 * cfg["r"] + 1, cfg["order"])
    return "%s: DVC %dx%dx%d synthetic volume, %d POIs, %d^3 subvolume, FFTCC3D->ICGN3D1" % (
        cfg_name, cfg["size"][0], cfg["size"][1], cfg["size"][2], cfg["n_poi"], 2 * cfg["r"] + 1)


def common_config(cfg_name, cfg, n_gpus):
    """The `config` object of the JSON line: identical in the GPU arm and the reference (CPU) arm."""
    return {"workload": workload_name(cfg_name, cfg), "pois_per_gpu": cfg["n_poi"], "conv": cfg["conv"], "stop": cfg["stop"],
            "parallelism": "GPU arm: POI shards over %d rank(s), one per GPU, no data-path collective; CPU arm: OpenMP threads of one host" % n_gpus,
            "l2": "GPU arm: flushed between timed steps (256 MiB write), timing = sum of per-step CUDA-event intervals; CPU arm: not applicable"}


# ---------------------------------------------------------------------------------------------------
def cpu_model():
    """CPU model string and logical core count of this host (BASELINE.md section 3 asks for both)."""
    model = "unknown"
    try:
        for line in open("/proc/cpuinfo"):
            if line.lower().startswith("model name"):
                model = line.split(":", 1)[1].strip()
                break
    except Exception:
        pass
    return model, os.cpu_count()


def pin_openmp():
    """Thread placement of the CPU arm: one thread per core, neighbours first.  Must be in the environment before the
    OpenMP runtime of the oracle library starts (it is loaded lazily, after this call)."""
    os.environ.setdefault("OMP_PROC_BIND", "close")
    os.environ.setdefault("OMP_PLACES", "cores")
    os.environ.setdefault("OMP_DYNAMIC", "false")


def time_cpu_path(cfg, ref, tar, pts, n_sample, repeats, threads):
    """The oracle port on `n_sample` evenly spaced POIs of the workload: ONE oracle object (image tables built once, like one
    set of reference DIC objects), `repeats` timed passes of FFT-CC + IC-GN after one untimed pass; the whole-workload time is
    prepare() once + per-POI stages scaled from the sample to all POIs.  Returns a dict with best-of-N and mean."""
    from oracle.oracle import Oracle2D, Oracle3D
    from opencorr_b200 import make_poi2d, make_poi3d
    kind, r, n = cfg["kind"], cfg["r"], cfg["n_poi"]
    sel = np.linspace(0, n - 1, n_sample).astype(np.int64)
    scale = n / float(n_sample)
    o = (Oracle2D if kind == "2d" else Oracle3D)(ref, tar, threads)
    t0 = time.perf_counter()
    o.prepare()
    t_prepare = time.perf_counter() - t0
    passes, q = [], None
    for rep in range(repeats + 1):
        q = make_poi2d(pts[sel]) if kind == "2d" else make_poi3d(pts[sel])
        t0 = time.perf_counter()
        if kind == "2d":
            o.fftcc2d(q, r, r)
            t1 = time.perf_counter()
            (o.icgn2d1 if cfg["order"] == 1 else o.icgn2d2)(q, r, r, cfg["conv"], cfg["stop"])
        else:
            o.fftcc3d(q, r, r, r)
            t1 = time.perf_counter()
            o.icgn3d1(q, r, r, r, cfg["conv"], cfg["stop"])
        t2 = time.perf_counter()
        if rep > 0:  # pass 0 warms caches / the OpenMP pool
            passes.append((t1 - t0, t2 - t1))
    whole = [t_prepare + scale * (a + b) for a, b in passes]
    best, mean = min(whole), sum(whole) / len(whole)
    model, ncpu = cpu_model()
    return {
        "value_best": n / best, "value_mean": n / mean, "ms_best": 1e3 * best, "ms_mean": 1e3 * mean, "passes": len(passes),
        "fftcc_s_best": min(a for a, _ in passes), "icgn_s_best": min(b for _, b in passes), "prepare_s": t_prepare,
        "n_sample": int(n_sample), "scale": scale, "threads": threads, "cpu_model": model, "logical_cpus": ncpu,
        "omp": {k: os.environ.get(k) for k in ("OMP_PROC_BIND", "OMP_PLACES")}, "queue": q, "sel": sel,
    }


def run_reference(args):
    """CPU arm: the oracle port of the reference on the host cores, all threads it would use."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    pin_openmp()
    from oracle.oracle import max_threads
    cfg, ref, tar, pts = make_workload(args.config, 0, 1)
    threads = max(1, max_threads() - 1)  # omp_get_num_procs() - 1, reference examples/test_2d_dic_fftcc_icgn1.cpp:40-41
    n_sample = min(cfg["n_poi"], args.cpu_sample if args.cpu_sample > 0 else (cfg["n_poi"] if cfg["kind"] == "2d" else 400))
    c = time_cpu_path(cfg, ref, tar, pts, n_sample, max(1, args.steps), threads)
    ms = c["ms_best"]
    value = c["value_best"]
    sample = ("%d of %d POIs of the workload per pass (evenly spaced); one oracle object, prepare() once (%.3f s) + per-POI stages x %.1f; "
              "best of %d passes after 1 warm-up pass (mean %.0f POI/s); %s, %d logical CPUs, %d OpenMP threads, OMP_PROC_BIND=%s OMP_PLACES=%s"
              % (n_sample, cfg["n_poi"], c["prepare_s"], c["scale"], c["passes"], c["value_mean"], c["cpu_model"], c["logical_cpus"], threads,
                 c["omp"]["OMP_PROC_BIND"], c["omp"]["OMP_PLACES"]))
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        # the same keys as the GPU arm's config
        "config": common_config(args.config, cfg, args.gpus),
        "reference_impl": "oracle port (oracle/oc_oracle.cpp); the reference itself needs Eigen/FFTW/OpenCV, absent here",
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample, "value_mean": c["value_mean"],
                         "cpu_model": c["cpu_model"], "logical_cpus": c["logical_cpus"]},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, c["queue"])
    print(json.dumps(line))
    return 0


# ---------------------------------------------------------------------------------------------------
def write_pgm(path, img):
    a = np.ascontiguousarray(img).astype(np.uint8)
    with open(path, "wb") as f:
        f.write(b"P5\n%d %d\n255\n" % (a.shape[1], a.shape[0]))
        f.write(a.tobytes())


def shim_e2e(cfg, ref, tar, steps, warmup, env_extra=None):
    """The step through the C++ shim (examples/shim_bench.cpp): the reference's class API on the caller's pageable memory."""
    binp = os.path.join(ROOT, "examples", "bin", "shim_bench")
    if cfg["kind"] != "2d" or not os.path.exists(binp) or float(np.abs(ref - np.round(ref)).max()) != 0.0:
        return None
    import tempfile
    d = tempfile.mkdtemp(prefix="ocb_bench_", dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
    try:
        write_pgm(os.path.join(d, "ref.pgm"), ref)
        write_pgm(os.path.join(d, "tar.pgm"), tar)
        x0, y0, nx, ny, sx, sy = cfg["grid"]
        cmd = [binp, os.path.join(d, "ref.pgm"), os.path.join(d, "tar.pgm")] + [str(v) for v in (x0, y0, nx, ny, sx, sy, cfg["r"], cfg["order"],
                                                                                    cfg["conv"], cfg["stop"], steps, warmup)]
        env = dict(os.environ)
        env.update(env_extra or {})
        out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=env)
        if out.returncode != 0:
            return {"error": (out.stderr or out.stdout).strip()[-300:]}
        rec = json.loads(out.stdout.strip().splitlines()[-1])
        ms = rec["ms"]
        mean = sum(ms) / len(ms)
        return {"value": rec["n_poi"] / (mean * 1e-3), "unit": UNIT, "ms_per_step": mean, "ms_min": min(ms), "n_poi": rec["n_poi"],
                "converged": rec["converged"], "first_step_incl_start_up_ms": rec["first_step_incl_start_up_ms"],
                "memory": "pageable (Image2D pixels, std::vector<POI2D>)", "devices": (env_extra or {}).get("OPENCORR_B200_DEVICES", "1"),
                "step": "FFTCC2D::compute + ICGN2D%d::prepare + compute on one pair (prepare() re-uploads the pair)" % cfg["order"]}
    finally:
        import shutil
        shutil.rmtree(d, ignore_errors=True)


def cold_start_record():
    try:
        out = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "cold_start_probe.py")], capture_output=True, text=True, timeout=300)
        rec = json.loads(out.stdout.strip().splitlines()[-1])
        rec["note"] = ("fresh process, C ABI; measured while this bench process keeps the GPU initialised (a first-ever process on an idle GPU "
                       "without persistence mode pays the driver's GPU initialisation on top)")
        return rec
    except Exception as e:  # noqa: BLE001
        return {"error": str(e)[:200]}


def group_e2e(ob, torch, devices, cfg_name, weak_ranks, steps, warmup, render_device):
    """One process, len(devices) GPUs, through a GROUP context of the C ABI (ocb_create_multi): host buffers in, host buffers
    out, the queue sharded inside the library.  weak_ranks > 0: the weak-scaling workload as ONE queue (the grids of that many
    ranks); 0: the config's own queue (strong scaling)."""
    cfg, ref, tar, pts = make_workload(cfg_name, 0, 1, device=render_device)
    if weak_ranks > 1:
        pts = np.concatenate([make_points(cfg_name, k) for k in range(weak_ranks)])
    kind, r = cfg["kind"], cfg["r"]
    n = len(pts)
    eng = ob.Engine(devices if len(devices) > 1 else devices[0])
    q0 = ob.make_poi2d(pts) if kind == "2d" else ob.make_poi3d(pts)
    h_ref, h_tar = torch.from_numpy(ref).pin_memory(), torch.from_numpy(tar).pin_memory()
    h_q0, h_q = torch.from_numpy(q0).pin_memory(), torch.empty((n, q0.shape[1]), dtype=torch.float32).pin_memory()

    def step():
        qn = h_q.numpy()
        if kind == "2d":
            eng._ck(eng._lib.ocb_set_images_2d(eng._ctx, h_ref.data_ptr(), h_tar.data_ptr(), ref.shape[1], ref.shape[0], 0))
            eng.fftcc2d(qn, r, r)
            eng.icgn2d_prepare()
            (eng.icgn2d1 if cfg["order"] == 1 else eng.icgn2d2)(qn, r, r, cfg["conv"], cfg["stop"])
        else:
            eng._ck(eng._lib.ocb_set_images_3d(eng._ctx, h_ref.data_ptr(), h_tar.data_ptr(), ref.shape[2], ref.shape[1], ref.shape[0]))
            eng.fftcc3d(qn, r, r, r)
            eng.icgn3d_prepare()
            eng.icgn3d1(qn, r, r, r, cfg["conv"], cfg["stop"])

    ts = []
    gc.collect()
    gc.disable()
    try:
        for i in range(warmup + steps):
            np.copyto(h_q.numpy(), h_q0.numpy())
            t0 = time.perf_counter()
            step()  # blocking like the reference's compute(): every member has synchronised when it returns
            if i >= warmup:
                ts.append(time.perf_counter() - t0)
    finally:
        gc.enable()
    res = h_q.numpy()
    zc = 16 if kind == "2d" else 18
    ms = 1e3 * sum(ts) / len(ts)
    eng.close()
    return {"workload": workload_name(cfg_name, dict(cfg, n_poi=n)), "devices": len(devices), "n_poi": n, "value": n / (ms * 1e-3), "unit": UNIT,
            "ms_per_step": ms, "ms_min": 1e3 * min(ts), "converged_frac": float((res[:, zc] >= 0).mean()),
            "h2d_bytes_per_step": int(len(devices) * (ref.nbytes + tar.nbytes) + 2 * q0.nbytes), "d2h_bytes_per_step": int(2 * q0.nbytes),
            "scaling": "weak" if weak_ranks else "strong"}


def make_points(cfg_name, rank):
    from opencorr_b200 import synth
    cfg = synth.CONFIGS[cfg_name]
    g = list(cfg["grid"])
    g[0] += rank
    return synth.grid_2d(*g) if cfg["kind"] == "2d" else synth.grid_3d(*g)


# ---------------------------------------------------------------------------------------------------
class ClockSampler:
    """Polls SM clock and throttle reasons through NVML from a thread DURING the timed region
    (nvidia-smi -lms cannot sample a region that lasts tens of milliseconds)."""

    def __init__(self, index, period_s=0.002):
        self.index, self.period = index, period_s
        self.samples, self.reasons = [], set()
        self.sm_max = None
        self._stop = False
        self._thread = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self._physical_index(index))
            self.sm_max = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nv = None

    @staticmethod
    def _physical_index(i):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            try:
                return int(vis.split(",")[i])
            except Exception:
                return i
        return i

    def _loop(self):
        nv = self.nv
        bits = {"hw_slowdown": nv.nvmlClocksEventReasonHwSlowdown if hasattr(nv, "nvmlClocksEventReasonHwSlowdown") else 0x8,
                "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}
        while not self._stop:
            try:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for name, bit in bits.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(self.period)

    def start(self):
        if self.nv is None:
            return
        import threading
        self._thread = threading.Thread(target=self._loop, daemon=True)
        self._thread.start()

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": self.sm_max, "reasons": []}
        if self._thread is None:
            return out
        self._stop = True
        self._thread.join(timeout=2)
        if self.samples:
            out["sm_mhz"] = statistics.median(self.samples)
            out["reasons"] = sorted(self.reasons)
            out["samples"] = len(self.samples)
        return out


def bind_to_gpu_numa_node(index):
    """Run this rank on the CPU cores next to its GPU (NVML's ideal-CPU set), before any host buffer is allocated: page-locked
    buffers then live in the memory of the socket the GPU's PCIe link hangs on, instead of crossing the inter-socket link on every
    copy.  One line of deployment hygiene for one-process-per-GPU jobs; returns a description for the JSON line."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(ClockSampler._physical_index(index))
        before = len(os.sched_getaffinity(0))
        pynvml.nvmlDeviceSetCpuAffinity(h)
        return "rank bound to the %d CPUs NVML lists for its GPU (of %d)" % (len(os.sched_getaffinity(0)), before)
    except Exception as e:  # noqa: BLE001
        return "not bound (%s)" % str(e)[:80]


def run_ours(args):
    import torch
    import torch.distributed as dist
    import opencorr_b200 as ob
    from opencorr_b200 import distributed as obd

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        print(json.dumps({"error": "no CUDA device; opencorr_b200 has no CPU fallback"}))
        return 2
    numa = bind_to_gpu_numa_node(local_rank) if world > 1 else "single rank: not bound"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    idle_group = None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
        idle_group = dist.new_group(backend="gloo")  # CPU-side barrier for the phases in which only rank 0 works
    if args.gpus != world and rank == 0:
        print("warning: --gpus %d but WORLD_SIZE=%d" % (args.gpus, world), file=sys.stderr)

    cfg, ref, tar, pts = make_workload(args.config, rank, world, device=dev)
    kind, r = cfg["kind"], cfg["r"]
    n = cfg["n_poi"]
    floats = 25 if kind == "2d" else 31
    eng = ob.Engine(local_rank)
    stream = torch.cuda.current_stream(dev)
    eng.set_stream(stream.cuda_stream)

    # ---------------- device-resident leg ("value") ----------------
    d_ref = torch.from_numpy(ref).to(dev)
    d_tar = torch.from_numpy(tar).to(dev)
    if world > 1:
        obd.broadcast_images(d_ref, d_tar, src=0)  # every rank renders the same pair; this is the NCCL path of the design
    q0 = (ob.make_poi2d(pts) if kind == "2d" else ob.make_poi3d(pts))
    d_q0 = torch.from_numpy(q0).to(dev)
    d_q = torch.empty_like(d_q0)
    if kind == "2d":
        eng.set_images_2d_dev(d_ref.data_ptr(), d_tar.data_ptr(), ref.shape[1], ref.shape[0])
    else:
        eng.set_images_3d_dev(d_ref.data_ptr(), d_tar.data_ptr(), ref.shape[2], ref.shape[1], ref.shape[0])
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)  # 256 MiB > 126 MB L2

    def step_resident(ev=None):
        d_q.copy_(d_q0)
        if kind == "2d":
            eng.fftcc2d_dev(d_q.data_ptr(), n, r, r)
            eng.icgn2d_prepare()
            if ev:
                ev[0].record(stream)
            (eng.icgn2d1_dev if cfg["order"] == 1 else eng.icgn2d2_dev)(d_q.data_ptr(), n, r, r, cfg["conv"], cfg["stop"])
            if ev:
                ev[1].record(stream)
        else:
            eng.fftcc3d_dev(d_q.data_ptr(), n, r, r, r)
            eng.icgn3d_prepare()
            if ev:
                ev[0].record(stream)
            eng.icgn3d1_dev(d_q.data_ptr(), n, r, r, r, cfg["conv"], cfg["stop"])
            if ev:
                ev[1].record(stream)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    for _ in range(args.warmup):
        step_resident()
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    launches0 = eng.launch_count()
    step_ms, icgn_ms = [], []
    wall0 = time.perf_counter()
    for _ in range(args.steps):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        step_resident((k0, k1))
        e1.record(stream)
        e1.synchronize()
        step_ms.append(e0.elapsed_time(e1))
        icgn_ms.append(k0.elapsed_time(k1))
    barrier()
    wall = time.perf_counter() - wall0
    launches = eng.launch_count() - launches0
    clocks = sampler.stop()
    total_ms = torch.tensor([sum(step_ms)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(total_ms, op=dist.ReduceOp.MAX)
    total_ms = float(total_ms.item())
    ms_per_step = total_ms / args.steps
    value = world * n / (ms_per_step * 1e-3)

    # iteration histogram / sanity of the last step
    res = d_q.cpu().numpy()
    zc, ic = (16, 17) if kind == "2d" else (18, 19)
    good = res[:, zc] >= 0
    hist = np.bincount(res[good, ic].astype(np.int64), minlength=int(cfg["stop"]) + 1).tolist()

    # ---------------- end-to-end leg ("e2e"): host buffers through the C ABI ----------------
    # Every rank is a caller with ITS OWN host buffers (pinned): the pair, its POI queue.  No collective: the path shards over
    # independent POIs, each GPU moves its data over its own PCIe link.
    h_ref = torch.from_numpy(ref).pin_memory()
    h_tar = torch.from_numpy(tar).pin_memory()
    h_q0 = torch.from_numpy(q0).pin_memory()
    h_q = torch.empty_like(h_q0).pin_memory()
    h_q0_np = h_q0.numpy()
    n_total = world * n
    img_bytes = ref.nbytes + tar.nbytes
    poi_bytes = q0.nbytes
    eng.use_own_stream()
    phases = []  # per-step host-side phase times (ms): set_images, (unused), FFTCC call, ICGN call

    def reset_queue():
        """The step's input: the pristine POI queue in pinned host memory.  Prepared OUTSIDE the timed region (the calls
        work in place on the caller's records, like the reference's compute(std::vector<POI2D>&)); a plain memcpy, because
        torch's copy_ fans 5 MB out over an OpenMP pool of ~127 threads and one straggler stalls it for tens of ms."""
        np.copyto(h_q.numpy(), h_q0_np)

    def step_e2e():
        # exactly what a caller of the reference API does: setImages, FFTCC compute, prepare, ICGN compute
        if kind == "2d":
            t = [time.perf_counter()]
            eng._ck(eng._lib.ocb_set_images_2d(eng._ctx, h_ref.data_ptr(), h_tar.data_ptr(), ref.shape[1], ref.shape[0], 0))
            t.append(time.perf_counter())
            qn = h_q.numpy()
            t.append(time.perf_counter())
            eng.fftcc2d(qn, r, r)
            t.append(time.perf_counter())
            eng.icgn2d_prepare()
            (eng.icgn2d1 if cfg["order"] == 1 else eng.icgn2d2)(qn, r, r, cfg["conv"], cfg["stop"])
            t.append(time.perf_counter())
            phases.append([1e3 * (b - a) for a, b in zip(t[:-1], t[1:])])
        else:
            eng._ck(eng._lib.ocb_set_images_3d(eng._ctx, h_ref.data_ptr(), h_tar.data_ptr(), ref.shape[2], ref.shape[1], ref.shape[0]))
            qn = h_q.numpy()
            eng.fftcc3d(qn, r, r, r)
            eng.icgn3d_prepare()
            eng.icgn3d1(qn, r, r, r, cfg["conv"], cfg["stop"])

    # warm-up: at least `warmup` steps AND ~0.2 s of wall clock -- on the pool's boxes one host-side stall of 60-80 ms
    # (seen inside a plain pinned-memory memcpy, i.e. not in this library) follows the pinned allocations above by
    # 20-50 ms; it must not land in the timed region
    # (count derived from the all-reduced resident step time, so every rank runs the same number of steps)
    n_w = int(min(100, max(3, args.warmup, math.ceil(200.0 / max(ms_per_step, 1e-3)))))
    for _ in range(n_w):
        reset_queue()
        step_e2e()
    barrier()
    # a generation-2 pass of Python's cyclic GC over the ~1e6 objects torch leaves on the heap takes 60-80 ms and used
    # to land in one of the timed steps; collect now and keep the collector off while timing (as timeit does)
    gc.collect()
    gc.disable()
    e2e_times = []
    for _ in range(args.steps):
        reset_queue()
        barrier()
        t0 = time.perf_counter()
        step_e2e()
        torch.cuda.synchronize(dev)
        e2e_times.append(time.perf_counter() - t0)
    gc.enable()
    e2e_ms = torch.tensor([1e3 * sum(e2e_times) / len(e2e_times)], dtype=torch.float64, device=dev)
    e2e_by_rank = [float(e2e_ms.item())]
    if world > 1:
        gathered = [torch.zeros_like(e2e_ms) for _ in range(world)]
        dist.all_gather(gathered, e2e_ms)
        e2e_by_rank = [float(t.item()) for t in gathered]
        dist.all_reduce(e2e_ms, op=dist.ReduceOp.MAX)
    e2e_ms = float(e2e_ms.item())
    e2e_value = n_total / (e2e_ms * 1e-3)
    e2e_sorted = sorted(1e3 * t for t in e2e_times)
    e2e_spread = {"min": e2e_sorted[0], "median": e2e_sorted[len(e2e_sorted) // 2], "max": e2e_sorted[-1],
                  "argmax_step": int(np.argmax(e2e_times))}
    if phases:
        ph = phases[-len(e2e_times):]
        e2e_spread["phases_ms_of_slowest_step[set_images,-,fftcc,icgn]"] = ph[int(np.argmax(e2e_times))]
        e2e_spread["phases_ms_median"] = [float(np.median([p[i] for p in ph])) for i in range(4)]
    h2d, d2h = world * (img_bytes + 2 * poi_bytes), world * 2 * poi_bytes  # whole job: every rank copies its own pair and queue

    # same end-to-end step with the images handed over as 8-bit arrays (what an image file holds; the
    # reference converts them to float on the host, src/oc_image.cpp:39,56): extra information, N=1 only
    e2e_u8 = None
    if world == 1 and float(np.abs(ref - np.round(ref)).max()) == 0.0 and ref.min() >= 0 and ref.max() <= 255:
        h8_ref = torch.from_numpy(ref.astype(np.uint8)).pin_memory()
        h8_tar = torch.from_numpy(tar.astype(np.uint8)).pin_memory()

        def step_e2e_u8():
            if kind == "2d":
                eng._ck(eng._lib.ocb_set_images_2d_u8(eng._ctx, h8_ref.data_ptr(), h8_tar.data_ptr(), ref.shape[1], ref.shape[0]))
                qn = h_q.numpy()
                eng.fftcc2d(qn, r, r)
                eng.icgn2d_prepare()
                (eng.icgn2d1 if cfg["order"] == 1 else eng.icgn2d2)(qn, r, r, cfg["conv"], cfg["stop"])
            else:
                eng._ck(eng._lib.ocb_set_images_3d_u8(eng._ctx, h8_ref.data_ptr(), h8_tar.data_ptr(), ref.shape[2], ref.shape[1], ref.shape[0]))
                qn = h_q.numpy()
                eng.fftcc3d(qn, r, r, r)
                eng.icgn3d_prepare()
                eng.icgn3d1(qn, r, r, r, cfg["conv"], cfg["stop"])

        for _ in range(max(3, args.warmup)):
            reset_queue()
            step_e2e_u8()
        ts = []
        gc.collect()
        gc.disable()
        for _ in range(args.steps):
            reset_queue()
            torch.cuda.synchronize(dev)
            t0 = time.perf_counter()
            step_e2e_u8()
            torch.cuda.synchronize(dev)
            ts.append(time.perf_counter() - t0)
        gc.enable()
        u8_ms = 1e3 * sum(ts) / len(ts)
        same = bool(np.array_equal(h_q.numpy()[:, :floats], res)) if False else None
        e2e_u8 = {"value": n / (u8_ms * 1e-3), "unit": UNIT, "ms_per_step": u8_ms,
                  "h2d_bytes_per_step": int(ref.size + tar.size + 2 * poi_bytes), "d2h_bytes_per_step": int(2 * poi_bytes)}

    # ---------------- roofline of the dominant kernel (IC-GN) ----------------
    peak, peak_src = load_peaks()
    icgn_avg_ms = sum(icgn_ms) / len(icgn_ms)
    bytes_per_launch = icgn_bytes_per_poi(kind, r) * n
    achieved = bytes_per_launch / (icgn_avg_ms * 1e-3) / 1e9
    traffic, ncu_pipes = None, None
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tp):
        try:
            rec = json.load(open(tp)).get(args.config, {})
            traffic = rec.get("icgn_dram_bytes_per_launch")
            if "ncu_issue_slots_busy_pct" in rec:  # the resources that actually bind (SURVEY 8(d)), from the committed ncu capture
                ncu_pipes = {"issue_slots_busy_pct": rec["ncu_issue_slots_busy_pct"], "fma_pipe_busy_pct": rec["ncu_fma_pipe_busy_pct"],
                             "shared_mem_pipe_busy_pct": rec["ncu_mem_pipes_busy_pct"], "source": rec.get("ncu_source")}
        except Exception:
            traffic, ncu_pipes = None, None
    roofline = {"bound": "hbm", "kernel": "icgn%s" % ("2d%d" % cfg["order"] if kind == "2d" else "3d1"), "achieved": achieved,
                "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                "algorithmic_bytes_per_poi": icgn_bytes_per_poi(kind, r), "kernel_ms": icgn_avg_ms,
                "kernel_share_of_step": icgn_avg_ms / (sum(step_ms) / len(step_ms)), "binding_resources_ncu": ncu_pipes,
                "note": "kernel is FP32-issue/shared-memory bound once tiles are on chip (DESIGN.md); the HBM fraction is reported as north_star asks"}

    # ---------------- CPU baseline on this box's host cores (rank 0, N=1 only) ----------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        pin_openmp()
        from oracle.oracle import max_threads
        threads = max(1, max_threads() - 1)
        n_sample = n if kind == "2d" else min(n, 300)
        c = time_cpu_path(cfg, ref, tar, pts, n_sample, 2, threads)
        qc, sel = c["queue"], c["sel"]
        # prepare() is paid once per image pair; the per-POI stages scale with the POI count, so the
        # whole-workload time is prepare + (fftcc + icgn) * n / n_sample
        cpu = {"value": c["value_best"], "unit": UNIT, "cores": threads, "kind": "port", "value_mean": c["value_mean"],
               "cpu_model": c["cpu_model"], "logical_cpus": c["logical_cpus"],
               "sample": "%d of %d POIs per pass, one oracle object; best of %d passes after 1 warm-up pass: fftcc %.3fs + prepare %.3fs + icgn %.3fs; "
                         "value = whole workload extrapolated (prepare once, per-POI stages x %.1f); OMP_PROC_BIND=%s OMP_PLACES=%s"
                         % (n_sample, n, c["passes"], c["fftcc_s_best"], c["prepare_s"], c["icgn_s_best"], c["scale"], c["omp"]["OMP_PROC_BIND"],
                            c["omp"]["OMP_PLACES"]),
               "value_compute_only": n_sample / (c["fftcc_s_best"] + c["icgn_s_best"])}
        # parity of the benchmarked run against the oracle on the sample (reported, not asserted)
        same = (res[sel, ic] == qc[:, ic]) & (res[sel, zc] >= 0) & (qc[:, zc] >= 0)
        cols = [2, 8] if kind == "2d" else [3, 7, 11]
        if same.any():
            cpu["parity_vs_gpu"] = {"n": int(len(sel)), "same_iteration": int(same.sum()),
                                    "max_abs_disp": float(np.abs(res[sel][same][:, cols] - qc[same][:, cols]).max()),
                                    "max_abs_zncc": float(np.abs(res[sel][same, zc] - qc[same, zc]).max())}

    # ---------------- rank 0 only: the shim, the group context, a cold start (the other ranks wait on the CPU) ----------------
    e2e_shim, capi_multi, cold = None, None, None
    torch.cuda.synchronize(dev)
    if rank == 0 and not args.no_extras:
        sub_steps = min(args.steps, 5)
        if world == 1:
            e2e_shim = shim_e2e(cfg, ref, tar, sub_steps, 2, {"OPENCORR_B200_DEVICE": str(local_rank)})
            cold = cold_start_record()
        capi_multi = {"note": "one process, %d device(s), GROUP context of the C ABI (ocb_create_multi); host buffers (pinned) in and out; "
                              "wall clock around the blocking calls" % world}
        if torch.cuda.device_count() >= world:
            devices = list(range(world))
            try:
                if world > 1:
                    capi_multi["weak_%s" % args.config] = group_e2e(ob, torch, devices, args.config, world, sub_steps, 2, dev)
                    if kind == "2d":
                        capi_multi["shim_weak_%s_pageable" % args.config] = shim_e2e(cfg, ref, tar, sub_steps, 2, {"OPENCORR_B200_DEVICES": ",".join(map(str, devices))})
                for name in ("C", "E", "D"):  # BASELINE.json configs[2], [4], [3]: whole queue on N devices (strong scaling; N = 1: one device)
                    if name != args.config or world > 1:
                        capi_multi["strong_%s" % name] = group_e2e(ob, torch, devices, name, 0, sub_steps, 2, dev)
            except Exception as e:  # noqa: BLE001
                capi_multi["error"] = str(e)[:300]
        else:
            capi_multi["skipped"] = "only %d of %d devices visible to rank 0" % (torch.cuda.device_count(), world)
    if idle_group is not None:
        dist.barrier(group=idle_group)

    if args.dump_outputs:
        dump_outputs(args.dump_outputs, res, rank, world)
    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": common_config(args.config, cfg, world),
            "wall_s_timed_region_incl_flush": wall,
            "cpu_binding": numa,
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h), "ms_per_step": e2e_ms,
                    "ms_per_step_by_rank": e2e_by_rank, "ms_per_step_spread_rank0": e2e_spread},
            "e2e_u8_images": e2e_u8,
            "e2e_shim": e2e_shim,
            "capi_multi": capi_multi,
            "cold_start": cold,
            "gpu_launches": int(launches),
            "roofline": roofline,
            "cpu_baseline": cpu,
            "results": {"converged_frac": float(good.mean()), "iteration_histogram": hist,
                        "fftcc_share_of_step": 1.0 - roofline["kernel_share_of_step"]},
        }
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    eng.close()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--config", default="B", choices=["A", "B", "C", "D", "E", "F"])
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--cpu-sample", type=int, default=0, help="POIs per step for --impl reference (0 = default)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the rank-0 extras (e2e_shim, capi_multi, cold_start)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the POI records of the last timed step to DIR/pois.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
