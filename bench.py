#!/usr/bin/env python
"""bench.py — the render hot path on N B200s, one process per GPU.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c1..c5] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one pass of the hot path over the workload: every scene of the named BASELINE configuration rendered
once at its full resolution / spp / depth.  Default workload: c5 = BASELINE.json configs[4] (3840x2160, 4.0M-triangle
mesh + 7 spheres + floor, 4096 spp) — the configuration `metric` is quoted on ("at 1/2/4/8 B200"), the BVH-traversal
path, and it fits one GPU.

  value   Mrays/s with the scene resident in HBM: ONE library call per scene (rrs_render_multi: sample split,
          persistent render kernel, ncclReduce at N > 1, resolve on rank 0) into a DEVICE image, CUDA events on the
          launching stream, max over ranks.
  e2e     the same call with a HOST image buffer on rank 0 (camera + parameters host->device, image device->host
          inside the timed region), wall clock, max over ranks.
  N > 1   STRONG scaling: the configuration's spp is split over the GPUs (rank g renders rrs_sample_range(g, N, spp)
          of every pixel), one reduce(sum) of the fp32 radiance buffers merges them (SURVEY.md 8e).
  extra   per_config: mini-records of the other BASELINE configurations (N = 1 only); parity_check: path census,
          NaN / negative pixels, and the N-GPU merged image against a single-GPU render of the same samples.
Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))
# stdout carries the one JSON line and nothing else: NCCL's own banner ("NCCL version ...") goes to stderr.  NCCL honours
# NCCL_DEBUG_FILE only above the VERSION level, where the banner is printed straight to stdout.
if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
    os.environ["NCCL_DEBUG"] = "WARN"
os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")

import numpy as np  # noqa: E402

METRIC = "Mrays/s (all bounces)"
UNIT = "Mrays/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=positive_int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c5", choices=["c1", "c2", "c3", "c4", "c5"])
    ap.add_argument("--spp", type=int, default=0, help="override the TOTAL spp (invalidates the headline; for experiments)")
    ap.add_argument("--e2e-steps", type=int, default=0, help="steps of the end-to-end leg (0 = max(3, steps // 4))")
    ap.add_argument("--no-per-config", action="store_true", help="skip the mini-records of the other configurations")
    ap.add_argument("--flags", type=int, default=0, help="RRS_FLAG_* for the timed renders (experiments)")
    ap.add_argument("--queue", type=int, default=0, help="rays in flight (0 = library default)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-seconds", type=float, default=15.0, help="target CPU time of the cpu_baseline sample")
    ap.add_argument("--ref-seconds", type=float, default=120.0, help="--impl reference: CPU time budget of the whole run")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the images of the last one as DIR/<scene>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs needs --impl ours: the reference arm sizes its spp from a timing probe, so its images differ "
                 "from run to run")
    return args


def positive_int(s):
    v = int(s)
    if v < 1:
        raise argparse.ArgumentTypeError(f"must be >= 1, got {v}")
    return v


DUMP_BYTES = 60 << 20    # below 64 MB in all, .npy headers included
DUMP_SEED = 0x5EEDB200


def dump_outputs(out_dir, named_images):
    """Write what the timed path returned to its caller in its last step: one (H, W, 3) float32 image per scene, as
    DIR/<scene>.npy.  An image larger than its share of DUMP_BYTES is written as a fixed, seeded sample of its pixels
    instead: DIR/<scene>.npy holds the (n, 3) sampled rows and DIR/<scene>_pixels.npy their flat pixel indices
    (row * W + column, ascending, float64).  The sample depends on the image size only, so two builds run with the
    same arguments are compared pixel for pixel."""
    out_dir = Path(out_dir)
    out_dir.mkdir(parents=True, exist_ok=True)
    share = DUMP_BYTES // max(1, len(named_images))
    for name, img in named_images:
        img = np.ascontiguousarray(img)
        if img.nbytes <= share:
            np.save(out_dir / f"{name}.npy", img)
            continue
        rows = img.reshape(-1, img.shape[-1])
        n = share // (rows.itemsize * rows.shape[1] + 8)
        idx = np.sort(np.random.default_rng(DUMP_SEED).choice(rows.shape[0], size=n, replace=False))
        np.save(out_dir / f"{name}.npy", rows[idx])
        np.save(out_dir / f"{name}_pixels.npy", idx.astype(np.float64))


def measured_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def bytes_per_ray_model(workload: str):
    """SURVEY.md 8(d): B_ray = 32*N_nodes + S_prim*N_prims + 144 + 64*P_miss (+16 per path).  The
    per-config constants are counted by the oracle offline (scripts/bytes_per_ray.py) and committed."""
    p = ROOT / "profiles" / "bytes_per_ray.json"
    if p.exists():
        d = json.loads(p.read_text())
        if workload in d:
            return d[workload]
    return None


COUNTERS_FILE = "profiles/r02_counters.json"


def kernel_counters(workload: str):
    """Per-ray constants of the render kernel measured by ncu on THIS command (`ncu ... python bench.py --workload X
    --spp S`, scripts/ncu_counters.py -> profiles/r02_counters.json): warp instructions, thread instructions and
    DRAM bytes per ray.  They are properties of the code and the workload (spp-invariant), so a launch's counts are
    these times its rays; the launch TIME is measured live."""
    p = ROOT / COUNTERS_FILE
    if p.exists():
        try:
            return json.loads(p.read_text()).get(workload)
        except Exception:
            return None
    return None


def roofline_block(workload, kname, rays, kernel_ms, n_launch, step_ms_total, clocks, sms, peak_hbm, peak_src):
    """The roofline of the render kernel.  Primary bound = the one that binds: thread-instruction issue
    (148 SMs x 128 lanes x SM clock).  The HBM figures ride along: the SURVEY 8(d) algorithmic-bytes model
    (`hbm_model`, an upper bound on traffic that an L2-resident scene never moves) and the measured DRAM bytes."""
    kms = max(kernel_ms, 1e-9)
    roof = {"bound": "issue", "kernel": kname, "achieved": None, "peak": None, "unit": "Tthread-inst/s", "frac": None,
            "traffic": None, "avg_launch_ms": kms / max(1, n_launch), "launches": n_launch,
            "share_of_step": kms / max(step_ms_total, 1e-9)}
    c = kernel_counters(workload)
    mhz = (clocks or {}).get("sm_mhz") or (clocks or {}).get("sm_max_mhz") or 1965.0
    roof["peak"] = sms * 128 * mhz * 1e6 / 1e12
    roof["peak_source"] = f"{sms} SMs x 128 lanes x {mhz:.0f} MHz (SM clock sampled during the timed region)"
    if c:
        ti = c["thread_inst_per_ray"] * rays
        wi = c["warp_inst_per_ray"] * rays
        roof["achieved"] = ti / (kms * 1e-3) / 1e12
        roof["frac"] = roof["achieved"] / roof["peak"]
        roof["warp_issue_frac"] = wi / (kms * 1e-3) / (sms * 4 * mhz * 1e6)
        roof["lanes_per_instruction"] = c["thread_inst_per_ray"] / c["warp_inst_per_ray"]
        roof["warp_inst_per_ray"] = c["warp_inst_per_ray"]
        roof["thread_inst_per_ray"] = c["thread_inst_per_ray"]
        roof["traffic"] = c["dram_bytes_per_ray"] * rays / max(1, n_launch)
        roof["dram"] = {"bytes_per_ray": c["dram_bytes_per_ray"], "achieved": c["dram_bytes_per_ray"] * rays / (kms * 1e-3) / 1e9,
                        "peak": peak_hbm, "unit": "GB/s", "frac": c["dram_bytes_per_ray"] * rays / (kms * 1e-3) / 1e9 / peak_hbm,
                        "peak_source": peak_src}
        roof["counters_source"] = c.get("source", COUNTERS_FILE)
        for k in ("l1tex_throughput_pct", "l1_global_load_sectors_per_ray", "l1_global_load_hit_pct", "l2_hit_pct", "issue_active_pct",
                  "long_scoreboard_stall_per_issue", "captured"):
            if k in c:
                roof[k] = c[k]
    model = bytes_per_ray_model(workload)
    if model:
        kb = model["kernel_bytes_per_ray"]
        b = kb["generate"] + kb["extend"] + kb["shade"]
        roof["hbm_model"] = {"bytes_per_ray": b, "achieved": rays * b / (kms * 1e-3) / 1e9, "peak": peak_hbm, "unit": "GB/s",
                             "frac": rays * b / (kms * 1e-3) / 1e9 / peak_hbm,
                             "note": "SURVEY 8(d) algorithmic bytes (32 B per visited node + 64 B per tested primitive + 144 B of "
                                     "queue state per ray) counted as if every byte came from HBM; the tree is L2-resident or "
                                     "shared-memory-resident, so these bytes are not moved: a model figure, not a bound"}
        roof["oracle_traversal"] = {"box_tests_per_ray": model["N_nodes"], "node_visits_per_ray": model["N_nodes"] / 2.0,
                                    "prims_tested_per_ray": model["N_prims"],
                                    "note": "ordered, t-pruned traversal of the exact-box reference tree, counted by the oracle"}
    return roof


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region.  In-process NVML (what nvidia-smi reads) on a
    thread, one sample every 2 ms, so that a timed region of ~100 ms still holds dozens of samples; an `nvidia-smi
    -lms` child process is the fallback when the NVML binding is missing (its start-up alone can outlast a short
    region, which is why it is not the first choice)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int, uuid: str | None = None):
        self.gpu = gpu_index
        self.proc = None
        self.path = None
        self.nvml = None
        self.handle = None
        self.thread = None
        self.running = False
        self.samples = []
        try:
            import pynvml
            pynvml.nvmlInit()
            h = None
            if uuid:
                try:
                    h = pynvml.nvmlDeviceGetHandleByUUID(uuid if uuid.startswith("GPU-") else "GPU-" + uuid)
                except Exception:
                    h = None
            if h is None:
                visible = os.environ.get("CUDA_VISIBLE_DEVICES", "")
                idx = gpu_index
                if visible:
                    ids = [v.strip() for v in visible.split(",") if v.strip()]
                    if gpu_index < len(ids) and ids[gpu_index].isdigit():
                        idx = int(ids[gpu_index])
                h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            self.nvml, self.handle = pynvml, h
        except Exception:
            self.nvml = None

    def _loop(self):
        nv, h = self.nvml, self.handle
        while self.running:
            try:
                mhz = float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                try:
                    why = int(nv.nvmlDeviceGetCurrentClocksEventReasons(h))
                except Exception:
                    why = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(h))
                self.samples.append((mhz, why))
            except Exception:
                pass
            time.sleep(0.002)

    def start(self):
        if self.nvml is not None:
            import threading
            self.running = True
            self.thread = threading.Thread(target=self._loop, daemon=True)
            self.thread.start()
            return
        try:
            f = tempfile.NamedTemporaryFile("w", suffix=".csv", delete=False)
            self.path = f.name
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu)], stdout=f, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0, "source": None}
        if self.nvml is not None:
            self.running = False
            if self.thread is not None:
                self.thread.join(timeout=2)
            nv = self.nvml
            bits = {"hw_slowdown": nv.nvmlClocksThrottleReasonHwSlowdown,
                    "hw_thermal_slowdown": nv.nvmlClocksThrottleReasonHwThermalSlowdown,
                    "sw_thermal_slowdown": nv.nvmlClocksThrottleReasonSwThermalSlowdown,
                    "sw_power_cap": nv.nvmlClocksThrottleReasonSwPowerCap}
            if self.samples:
                seen = 0
                for _, why in self.samples:
                    seen |= why
                out.update(sm_mhz=float(np.median([m for m, _ in self.samples])), sm_max_mhz=self.max_mhz,
                           reasons=sorted(k for k, b in bits.items() if seen & b), samples=len(self.samples), source="nvml")
            return out
        if self.proc is None:
            return out
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        try:
            for line in Path(self.path).read_text().splitlines():
                f = [x.strip() for x in line.split(",")]
                if len(f) < 9:
                    continue
                try:
                    sm.append(float(f[1]))
                    mx.append(float(f[2]))
                except ValueError:
                    continue
                for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], f[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), reasons=sorted(reasons), samples=len(sm),
                       source="nvidia-smi")
        return out


# ---------------------------------------------------------------------------------------------
# reference arm: the reference's own CPU implementation of the path, timed on the host cores.
# The Rust crate cannot be built in this image (no cargo/rustc), so it is the oracle port.
# ---------------------------------------------------------------------------------------------
def cpu_scenes(specs, hdri):
    """The oracle's scenes of a workload, built ONCE (the restated reference build of the 4M-triangle tree takes about a
    minute; like the reference's own timer, main.rs:59-100, the samples below time the tile loop only)."""
    import oracle
    return [(spec, oracle.OracleScene(spec.tables(), hdri.pixels, heuristic=(spec.heuristic.kind, spec.heuristic.splits), build_mode=1),
             oracle.camera_new(**spec.camera_args)) for spec in specs]


def cpu_render_sample(cfg, scenes_, spp, threads):
    """Render every scene of the workload at `spp` samples with the oracle; returns (rays, seconds)."""
    import oracle
    rays, secs = 0, 0.0
    for spec, osc, cam17 in scenes_:
        _, st = osc.render(cam17, cfg.width, cfg.height, spp, max_bounces=cfg.max_bounces, rng_mode=oracle.RNG_WIDE, nthreads=threads)
        rays += st["rays"]
        secs += st["seconds"]  # the tile loop only, like rayrs/src/main.rs:59-100
    return rays, secs


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import oracle
    from rayrs_b200 import scenes
    oracle.build()
    cfg = scenes.CONFIGS[args.workload]
    specs = cfg.specs()
    hdri = scenes.synthetic_hdri(2048, 1024)
    threads = oracle.hardware_threads()
    osc = cpu_scenes(specs, hdri)
    # size the per-step sample from a 1-spp probe so that the whole run ends within a few minutes
    r1, s1 = cpu_render_sample(cfg, osc, 1, threads)
    budget = args.ref_seconds / max(1, args.steps + args.warmup)
    spp = int(max(1, min(cfg.spp, budget / max(s1, 1e-3))))
    for _ in range(args.warmup):
        cpu_render_sample(cfg, osc, spp, threads)
    rays, secs = 0, 0.0
    for _ in range(args.steps):
        r, s = cpu_render_sample(cfg, osc, spp, threads)
        rays += r
        secs += s
    value = rays / secs / 1e6
    sample = f"{args.workload}: all {len(specs)} scene(s) at {cfg.width}x{cfg.height}, {spp} of {cfg.spp} spp per step (Mrays/s is spp-invariant)"
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": secs / max(1, args.steps) * 1e3, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": cfg.description, "scenes": [s.name for s in specs], "width": cfg.width, "height": cfg.height,
                   "spp_total": cfg.spp, "max_bounces": cfg.max_bounces, "hdri": "synthetic 2048x1024",
                   "spp_per_step": spp, "cpu_threads": threads,
                   "note": "restated reference (oracle port, g++ -O3 -ffp-contract=off), not the Rust binary: no Rust toolchain in "
                           "the image; each step renders a bounded sample of the workload (spp_per_step of spp_total samples per "
                           "pixel at full resolution; Mrays/s is spp-invariant)"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------
KERNEL_NAMES = {0: "k_wavefront", 1: "k_generate/k_extend/k_shade", 2: "k_pathloop"}


def run_ours(args):
    import torch
    import torch.distributed as dist
    from rayrs_b200 import _ffi, api, scenes

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — rayrs_b200 has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    # ---- the library's communicator: rank 0 makes the NCCL id, torch.distributed only carries its 128 bytes ----
    def exchange(raw):
        box = [raw]
        dist.broadcast_object_list(box, src=0)
        return box[0]

    if world > 1:
        comm = api.Comm(world, rank, local, exchange)
        comm_ptr = comm.ptr
    else:
        comm = None
        comm_ptr = C.c_void_p()
        devs = (C.c_int * 1)(local)
        _ffi.check(_ffi.cuda_lib().rrs_comm_init_all(devs, 1, C.byref(comm_ptr)))

    cfg = scenes.CONFIGS[args.workload]
    spp_total = args.spp or cfg.spp          # strong scaling: the configuration's spp, split over the ranks
    first, count = api.sample_range(rank, world, spp_total)
    specs = cfg.specs()
    hdri = scenes.synthetic_hdri(2048, 1024)
    # the process's CUDA start-up (context creation on this device) is paid once per process whatever the scene: timed on
    # its own so that scene_setup_s below is the scene's setup, not the driver's
    t_cuda = time.time()
    torch.zeros(1, device=dev)
    torch.cuda.synchronize(dev)
    t_cuda = time.time() - t_cuda
    t_setup = time.time()
    built = [(spec, spec.scene(hdri, device=local, with_f64=False, device_build=True, topology=False), spec.camera()) for spec in specs]
    t_setup = time.time() - t_setup
    build_s = sum(sc.build_seconds for _, sc, _ in built)
    build_timing = [sc.build_timing for _, sc, _ in built]
    W, H = cfg.width, cfg.height
    stream = torch.cuda.current_stream(dev)
    sptr = stream.cuda_stream
    out = [torch.empty((H, W, 3), dtype=torch.float32, device=dev) for _ in built] if rank == 0 else [None] * len(built)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2
    sms = torch.cuda.get_device_properties(dev).multi_processor_count

    def render(sc, cam, spp, out_ptr, out_is_device, flags=0, max_bounces=None):
        """ONE library call: sample split over the ranks of the communicator, render, reduce, resolve on rank 0"""
        api.render_multi(cam, [sc.handle], comm_ptr, spp, cfg.max_bounces if max_bounces is None else max_bounces,
                         out_ptr=out_ptr, out_is_device=out_is_device, streams=[sptr], queue_capacity=args.queue, flags=flags)

    def step_device(flags=0):
        """inputs resident in HBM, image stays on the device; returns (rays, launches, stats of the last scene)"""
        rays = launches = 0
        kernel_ms = 0.0
        st = None
        flush.fill_(1)  # L2 flush between timed iterations (inside the region: ~0.1 ms); a torch kernel, not counted
        for k, (spec, sc, cam) in enumerate(built):
            render(sc, cam, spp_total, out[k].data_ptr() if rank == 0 else 0, True, flags)
            st = sc.stats()                      # waits for this rank's part
            rays += st["rays"]
            launches += st["kernel_launches"]    # OUR render + resolve kernels and NCCL's reduce; torch's fill_ is not counted
            kernel_ms += st["device_ms"]
        return rays, launches, kernel_ms, st

    # the caller's image buffers, page-locked (the library DMAs straight into a pinned destination)
    host_pin = [torch.empty((H, W, 3), dtype=torch.float32, pin_memory=True) for _ in built] if rank == 0 else []

    def step_e2e():
        """the public call with a HOST image on rank 0: camera + parameters host->device, image device->host"""
        rays = 0
        for k, (spec, sc, cam) in enumerate(built):
            render(sc, cam, spp_total, host_pin[k].data_ptr() if rank == 0 else 0, False, args.flags)
            rays += sc.stats()["rays"]
        return rays

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # ---- device-resident timing -----------------------------------------------------------
    sampler = None
    if rank == 0:
        try:
            uuid = str(torch.cuda.get_device_properties(dev).uuid)
        except Exception:
            uuid = None
        sampler = ClockSampler(local, uuid)  # NVML is initialised here, outside the timed region
    warmup = max(3, args.warmup)
    for _ in range(warmup):
        step_device(args.flags)
    barrier()
    if sampler is not None:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    rays = launches = 0
    kernel_ms = 0.0
    last = None
    for _ in range(args.steps):
        r, l, km, last = step_device(args.flags)
        rays += r
        launches += l
        kernel_ms += km
    e1.record(stream)
    barrier()
    ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    tot = torch.tensor([float(rays), float(launches)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    clocks = sampler.stop() if sampler is not None else None
    ms_total = float(ms.item())
    rays_all, launches_all = float(tot[0].item()), int(tot[1].item())
    census = {k: int(last[k]) for k in ("census_mismatch_pixels", "nan_pixels", "negative_pixels")} if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, [(spec.name, out[k].cpu().numpy()) for k, (spec, _, _) in enumerate(built)])

    # ---- end to end ---------------------------------------------------------------------------
    e2e_steps = args.e2e_steps or max(3, args.steps // 4)
    for _ in range(2):
        step_e2e()
    barrier()
    t0 = time.perf_counter()
    rays_e2e = 0
    e2e_step_ms = []
    for _ in range(e2e_steps):
        ts = time.perf_counter()
        rays_e2e += step_e2e()
        e2e_step_ms.append((time.perf_counter() - ts) * 1e3)
    barrier()
    e2e_s = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
    e2e_r = torch.tensor([float(rays_e2e)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
        dist.all_reduce(e2e_r, op=dist.ReduceOp.SUM)

    # ---- parity check carried in the line: the N-GPU merged image against ONE GPU rendering the same samples ----
    # (collective: every rank joins the split render; rank 0 then renders the same 8 spp alone through rrs_render)
    check_spp = 8
    spec0, sc0, cam0 = built[0]
    chk = torch.empty((H, W, 3), dtype=torch.float32, device=dev) if rank == 0 else None
    render(sc0, cam0, check_spp, chk.data_ptr() if rank == 0 else 0, True)
    sc0.stats()
    parity = None
    if rank == 0:
        st_multi = sc0.stats()
        solo = api.render_gpu(cam0, sc0, check_spp, cfg.max_bounces, out=np.empty((H, W, 3), dtype=np.float32),
                              queue_capacity=args.queue)
        a = chk.cpu().numpy().astype(np.float64)
        b = solo.astype(np.float64)
        rel = np.abs(a - b) / (np.abs(b) + 1e-3)
        parity = {"timed_steps": census,
                  "split_vs_single_gpu": {"scene": spec0.name, "spp": check_spp, "n_gpus": world,
                                          "max_rel_diff": float(rel.max()), "mean_rel_diff": float(rel.mean()),
                                          "census_mismatch_pixels": int(st_multi["census_mismatch_pixels"]),
                                          "tolerance": 1e-4},
                  "ok": bool(census["census_mismatch_pixels"] == 0 and census["nan_pixels"] == 0 and census["negative_pixels"] == 0
                             and st_multi["census_mismatch_pixels"] == 0 and rel.max() <= 1e-4)}
    barrier()

    # ---- traversal counters of this workload (COUNT form of the kernel, reduced spp; BVH scenes only) ----
    trav = None
    if rank == 0 and any(sc.n_prims > 8 for _, sc, _ in built):
        nv = pt = rr = 0
        for spec, sc, cam in built:
            tmp = torch.zeros((H, W, 4), dtype=torch.float32, device=dev)
            api.render_accumulate(cam, sc, 2, cfg.max_bounces, tmp.data_ptr(), sptr, spp_total=2, queue_capacity=args.queue,
                                  flags=_ffi.RRS_FLAG_COUNT_TRAVERSAL)
            st = sc.stats()
            nv += st["nodes_visited"]
            pt += st["prims_tested"]
            rr += st["rays"]
            del tmp
        trav = {"node_visits_per_ray": nv / max(1, rr), "box_tests_per_ray": 2.0 * nv / max(1, rr), "prims_tested_per_ray": pt / max(1, rr),
                "sample": "2 spp, RRS_FLAG_COUNT_TRAVERSAL"}
    barrier()

    # ---- mini-records of the other configurations (N = 1) -------------------------------------
    per_config = None
    if world == 1 and not args.no_per_config:
        per_config = {}
        peak, peak_src = measured_peaks()
        for key in ("c1", "c2", "c3", "c4"):
            if key == args.workload:
                continue
            try:
                per_config[key] = mini_record(key, scenes, api, _ffi, torch, dev, sptr, hdri, flush, clocks, sms, peak, peak_src, args)
            except Exception as e:  # a mini-record must not take the headline down
                per_config[key] = {"error": repr(e)}

    if rank == 0:
        value = rays_all / (ms_total * 1e-3) / 1e6
        e2e_value = float(e2e_r.item()) / float(e2e_s.item()) / 1e6
        peak, peak_src = measured_peaks()
        kname = KERNEL_NAMES.get(int(last["kernel_form"]), "?")
        # the dominant kernel is the one persistent render kernel (one launch per scene render); its launch durations
        # are the CUDA-event times around it on the launching stream (RrsStats.device_ms), measured live above
        roof = roofline_block(args.workload, kname, rays, kernel_ms, args.steps * len(built), ms_total, clocks, sms, peak, peak_src)
        if trav:
            roof["gpu_traversal"] = trav
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            import oracle  # cpu_baseline leg: the one place bench.py may execute oracle/
            oracle.build()
            threads = oracle.hardware_threads()
            osc = cpu_scenes(specs, hdri)
            r1, s1 = cpu_render_sample(cfg, osc, 1, threads)
            s_spp = int(max(1, min(cfg.spp, args.cpu_seconds / max(s1, 1e-3))))
            r, s = cpu_render_sample(cfg, osc, s_spp, threads) if s_spp > 1 else (r1, s1)
            cpu = {"value": r / s / 1e6, "unit": UNIT, "cores": threads, "kind": "port",
                   "sample": f"{args.workload}: all {len(specs)} scene(s) at {W}x{H}, {s_spp} of {cfg.spp} spp, {r} rays in {s:.1f} s"}
        cam_bytes = (len(bytes(_ffi.RrsCamera())) + len(bytes(_ffi.RrsRenderParams()))) * len(built)
        spp_note = "" if not args.spp else f" [total spp overridden to {spp_total}]"
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": warmup,
            "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": cfg.description + spp_note,
                       "scenes": [s.name for s in specs], "width": W, "height": H, "spp_total": spp_total,
                       "spp_per_gpu": [api.sample_range(r_, world, spp_total)[1] for r_ in range(world)],
                       "primitives": [sc.n_prims for _, sc, _ in built], "bvh_nodes": [sc.n_nodes for _, sc, _ in built],
                       "max_bounces": cfg.max_bounces, "hdri": "synthetic 2048x1024",
                       "parallelism": f"sample-split x{world} inside rrs_render_multi, one ncclReduce(sum) of the fp32 radiance buffer",
                       "l2": "256 MB L2 flush between steps (inside the timed region)",
                       "rays_per_step": rays_all / args.steps, "scene_setup_s": t_setup, "cuda_startup_s": t_cuda, "bvh_build_s": build_s,
                       "bvh_build": "same-tree build on the device (rrs_bvh_build), numbering + flattening on the host", "bvh_build_timing_s": build_timing},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": cam_bytes,
                    "d2h_bytes_per_step": W * H * 3 * 4 * len(built), "steps": e2e_steps, "ms_per_step": e2e_step_ms,
                    "with_setup": {"value": float(e2e_r.item()) / e2e_steps / (float(e2e_s.item()) / e2e_steps + t_setup) / 1e6, "unit": UNIT,
                                   "note": "one step plus the scene setup of this run (mesh load + host BVH build + upload), "
                                           "which the reference's timer excludes (main.rs:59-100)"}},
            "gpu_launches": launches_all,
            "clocks": clocks,
            "roofline": roof,
            "phases_ms": {k: float(last[k]) for k in ("generate_ms", "extend_ms", "shade_ms")} | {"iterations": int(last["iterations"]),
                          "note": "last timed launch; shares from in-kernel cycle counters"},
            "cpu_baseline": cpu,
            "extra": {"parity_check": parity, "per_config": per_config},
        }
        print(json.dumps(line), flush=True)
    for _, sc, _ in built:
        sc.close()
    if comm is not None:
        comm.close()
    else:
        _ffi.cuda_lib().rrs_comm_destroy(comm_ptr)
    if world > 1:
        dist.destroy_process_group()


def mini_record(key, scenes, api, _ffi, torch, dev, sptr, hdri, flush, clocks, sms, peak, peak_src, args, steps=2):
    """One BASELINE configuration at full size on one GPU: 1 warm-up + `steps` timed steps (L2 flushed), device-resident."""
    cfg = scenes.CONFIGS[key]
    specs = cfg.specs()
    t0 = time.time()
    built = [(spec, spec.scene(hdri, device=dev.index, with_f64=False, device_build=True, topology=False), spec.camera()) for spec in specs]
    setup = time.time() - t0
    W, H = cfg.width, cfg.height
    acc = torch.zeros((H, W, 4), dtype=torch.float32, device=dev)
    img = torch.empty((H, W, 3), dtype=torch.float32, device=dev)
    stream = torch.cuda.current_stream(dev)

    def step():
        rays, kms, st = 0, 0.0, None
        flush.fill_(1)
        for spec, sc, cam in built:
            acc.zero_()
            api.render_accumulate(cam, sc, cfg.spp, cfg.max_bounces, acc.data_ptr(), sptr, spp_total=cfg.spp)
            api.resolve(sc, acc.data_ptr(), W, H, cfg.spp, img.data_ptr(), True, sptr)
            st = sc.stats()
            rays += st["rays"]
            kms += st["device_ms"]
        return rays, kms, st

    step()
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    rays = 0
    kms = 0.0
    st = None
    for _ in range(steps):
        r, k, st = step()
        rays += r
        kms += k
    e1.record(stream)
    torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1)
    rec = {"workload": cfg.description, "value": rays / (ms * 1e-3) / 1e6, "unit": UNIT, "ms_per_step": ms / steps, "steps": steps,
           "rays_per_step": rays / steps, "scene_setup_s": setup,
           "census_mismatch_pixels": int(st["census_mismatch_pixels"]), "nan_pixels": int(st["nan_pixels"]),
           "roofline": roofline_block(key, KERNEL_NAMES.get(int(st["kernel_form"]), "?"), rays, kms, steps * len(built), ms, clocks, sms, peak, peak_src)}
    if any(sc.n_prims > 8 for _, sc, _ in built):
        nv = pt = rr = 0
        for spec, sc, cam in built:
            acc.zero_()
            api.render_accumulate(cam, sc, 2, cfg.max_bounces, acc.data_ptr(), sptr, spp_total=2, flags=_ffi.RRS_FLAG_COUNT_TRAVERSAL)
            s2 = sc.stats()
            nv += s2["nodes_visited"]
            pt += s2["prims_tested"]
            rr += s2["rays"]
        rec["roofline"]["gpu_traversal"] = {"node_visits_per_ray": nv / max(1, rr), "box_tests_per_ray": 2.0 * nv / max(1, rr),
                                            "prims_tested_per_ray": pt / max(1, rr), "sample": "2 spp, RRS_FLAG_COUNT_TRAVERSAL"}
    for _, sc, _ in built:
        sc.close()
    return rec


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
