#!/usr/bin/env python
"""bench.py -- headline benchmark of the tinsel_b200 path tracer (see BASELINE.json).

    python bench.py --gpus N --steps K --warmup W            # our arm (one process per GPU under torchrun)
    python bench.py --impl reference --gpus N --steps K --warmup W   # reference CPU arm

Metric: Msamples/s (camera paths incl. all bounces and shadow rays per second), whole job.
Workload: BASELINE.json configs[1] = data/cornell.tin, 1024x1024, Gaussian filter, maxDepth 4;
a "step" is one pass of the hot path adding SPP_PER_STEP samples to every pixel of the image.

`value`   device-resident: scene and accumulator in HBM, timed with CUDA events on the launching
          stream (an explicit torch stream handed to tb200_set_stream), max over ranks.  N > 1: image
          rows are sharded over the N ranks (interleaved 4-row tile rows, fixed total work => "strong"
          scaling) and the accumulated radiance is summed onto rank 0 with one NCCL reduce inside the
          timed region.
`e2e`     the same metric through the reference-facing call, tb200_render() = Renderer::Render:
          1 spp per call, HOST output buffer, device->host copy of the whole frame inside every call,
          host clock.  N > 1: ONE multi-device renderer (tb200_create_multi, what the plugin creates
          for TINSEL_GPUS=N) driven by rank 0 over all N GPUs -- row slabs, every GPU copies its own
          rows to the host over its own PCIe link, no reduce -- while the other ranks wait on a
          host-side (gloo) barrier.
`configs` (N = 1) the other BASELINE.json GPU configurations at their own sizes, same measurements.
`gpu_baseline` the reference's own GPU megakernel (src/render.cu, compiled for sm_100a with its
          Release flags into oracle/_ref) on the same GPU: the secondary bar of SURVEY.md 2b.
"""
import argparse
import ctypes as C
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# BASELINE.json configs: (scene, width, height, spp per step); cornell = configs[1] is the bench workload
MAIN = ("cornell", 1024, 1024, 32)
OTHER_WORKLOADS = {"ajax": (1024, 1024, 16), "veach": (1920, 1080, 16), "env": (2048, 2048, 16)}
E2E_CALLS_PER_STEP = 8          # Render() calls (1 spp each) per e2e step
CPU_SPP = 8                     # spp per step of the CPU arm (bounded sample of the workload)

# Algorithmic bytes per camera sample, counted on the REFERENCE traversal order by the instrumented
# oracle (tools/count_bytes.py; formula of SURVEY.md 8d, restated in DESIGN.md), plus per-kernel
# constants read off the committed ncu captures (instructions per sample, lanes, DRAM bytes,
# traversal share of the kernel's time): tools/algo_bytes.json names the capture each comes from.
ALGO_JSON = os.path.join(ROOT, "tools", "algo_bytes.json")


def load_algo(scene):
    with open(ALGO_JSON) as f:
        return json.load(f)["scenes"][scene]


def read_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)", float(d.get("sm_max_mhz", 1965.0))
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)", 1965.0


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons while the timed region runs (nvidia-smi equivalent via NVML)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self.stop_flag = False
        self.ok = False

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            names = {
                nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
                nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap",
                nv.nvmlClocksThrottleReasonHwPowerBrakeSlowdown: "hw_power_brake",
            }
            self.ok = True
            while not self.stop_flag:
                self.samples.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
                time.sleep(0.05)
        except Exception as e:  # noqa: BLE001
            self.error = str(e)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["unavailable"]}
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2], "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


def workload_config(scene, w, h, spp, n_gpus):
    return {
        "workload": "tinsel data/%s.tin %dx%d, Gaussian filter, maxDepth from the scene file, %d spp per step" % (scene, w, h, spp),
        "scene": "scenes/%s.tsnap (snapshot of the reference loader's Scene)" % scene,
        "width": w, "height": h, "spp_per_step": spp,
        "sharding": ("value: interleaved 4-row tile rows over %d rank(s), one NCCL sum-reduce of the accumulator; "
                     "e2e: one multi-device renderer, contiguous row slabs, each GPU copies its own rows to the host") % n_gpus
                    if n_gpus > 1 else "single GPU",
        "l2": "flushed between timed steps (256 MiB device write outside the per-step events)",
    }


# ---------------------------------------------------------------------------------------------------
# CPU arm: the reference's own CPU implementation (oracle/_ref = tinsel src/render.cpp compiled
# unmodified, literal glibc flavour) with the per-sample-seeded work-stealing driver (ref_render_pool)
# ---------------------------------------------------------------------------------------------------
def host_threads():
    """Threads for the CPU arm: the cores this container may actually use.  os.cpu_count() reports the
    host's 128 logical CPUs, but the box runs under a cgroup CPU quota (cpu.max = 16 CPUs on this pool):
    128 threads on 16 CPUs measured 5.4 Msamples/s against 12.7 with 32 (tools/cpu_scaling.py), so
    the arm uses twice the quota (both hardware threads of each core's worth), capped by the CPU count."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except (AttributeError, OSError):
        pass
    for path in ("/sys/fs/cgroup/cpu.max",):
        try:
            quota, period = open(path).read().split()[:2]
            if quota != "max":
                n = min(n, max(1, int(2 * int(quota) / int(period))))
        except (OSError, ValueError):
            pass
    try:
        q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
        p = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
        if q > 0:
            n = min(n, max(1, int(2 * q / p)))
    except (OSError, ValueError):
        pass
    return n


class CpuArm:
    def __init__(self, scene, w, h):
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import refdrv
        import tinsel_b200 as tb
        self.w, self.h = w, h
        self.threads = host_threads()
        if refdrv.have_ref("literal"):
            self.kind = "reference"
            self.sc = refdrv.RefScene.from_snapshot(tb.scene_path(scene), "literal")
            self.sc.set_size(w, h)
            self.render = lambda f0, n: self.sc.render_pool(f0, n, self.threads)
        else:
            import subprocess
            self.kind = "port"
            subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "oracle"), "port"])
            self.sc = refdrv.PortScene.from_snapshot(tb.scene_path(scene))
            self.sc.set_size(w, h)
            self.render = lambda f0, n: self.sc.render_seeded(f0, n, self.threads)

    def warm(self):
        # idle host cores (a VM's vCPUs in particular) take a while to come up: the first calls of a
        # process measured 3-5x below the steady state on the same box
        t0 = time.time()
        while time.time() - t0 < 1.5:
            self.render(1000, 1)

    def timed(self, spp):
        t0 = time.time()
        self.render(0, spp)
        dt = time.time() - t0
        return self.w * self.h * spp / dt / 1e6, dt

    def close(self):
        self.sc.close()


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    scene, w, h, spp = MAIN
    arm = CpuArm(scene, w, h)
    arm.warm()
    vals = []
    for i in range(args.warmup + args.steps):
        msps, dt = arm.timed(CPU_SPP)
        if i >= args.warmup:
            vals.append(dt)
    total_dt = sum(vals)
    value = w * h * CPU_SPP * len(vals) / total_dt / 1e6
    line = {
        "impl": "reference",
        "metric": "Msamples/sec (paths x spp / s)", "value": value, "unit": "Msamples/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": total_dt / len(vals) * 1e3, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic (scene snapshot, random paths)",
        "config": workload_config(scene, w, h, spp, args.gpus),
        "cpu_baseline": {"value": value, "unit": "Msamples/s", "cores": arm.threads, "kind": arm.kind,
                         "sample": "%dx%d image, %d spp per step, per-sample-seeded work-stealing driver (4-row strips) over the "
                                   "reference's PathTrace/AddSample" % (w, h, CPU_SPP)},
        "e2e": {"value": value, "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    arm.close()
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------------
def roofline_block(scene, value_msps, avg_launch_s, per_launch_samples, sm_mhz):
    """HBM roofline on algorithmic bytes (the contract's form) next to the bound that actually binds."""
    algo = load_algo(scene)
    peak, peak_src, sm_max = read_peaks()
    ncu = algo.get("ncu", {})
    achieved = algo["bytes_per_sample"] * per_launch_samples / avg_launch_s / 1e9
    out = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
           "traffic": ncu.get("dram_bytes_per_sample") and ncu["dram_bytes_per_sample"] * per_launch_samples,
           "traffic_source": ncu.get("source"),
           "kernel": ncu.get("kernel", "k_wavefront2"), "peak_source": peak_src,
           "algorithmic_bytes_per_sample": algo["bytes_per_sample"],
           "traversal_bytes_per_sample": algo.get("traversal_bytes_per_sample")}
    share = ncu.get("traversal_share")
    # scenes that live in shared memory move (almost) no bytes at all: an HBM fraction of their traversal would
    # only be a large meaningless number, so it is not printed; `frac` above stays, per the contract, flagged
    out["hbm_frac_is_a_bound"] = not algo.get("on_chip", False)
    if share and not algo.get("on_chip", False):
        # SURVEY 8d: traversal bytes over the traversal share of the kernel's time
        trav = algo["traversal_bytes_per_sample"] * per_launch_samples / (avg_launch_s * share) / 1e9
        out["traversal"] = {"achieved": trav, "frac": trav / peak, "share_of_kernel_time": share}
    ips = ncu.get("inst_per_sample")
    if ips:
        clock = (sm_mhz or sm_max) * 1e6
        peak_issue = 148 * 4 * clock                      # warp instructions per second, 4 schedulers per SM
        got = ips * value_msps * 1e6
        out["issue"] = {"achieved_ginst_s": got / 1e9, "peak_ginst_s": peak_issue / 1e9, "frac": got / peak_issue,
                        "inst_per_sample": ips, "lanes_per_inst": ncu.get("lanes"),
                        "lane_frac": got / peak_issue * (ncu.get("lanes") or 32.0) / 32.0}
    out["binding"] = algo.get("binding", "issue slots / dependent-load latency, not HBM")
    out["note"] = ("algorithmic bytes on the reference traversal order; the working set is SMEM/L2 resident "
                   "(`traffic` = measured DRAM bytes), so `frac` is throughput relative to streaming those bytes "
                   "from HBM, not HBM utilisation; `issue.frac` is the fraction of the SMs' issue slots in use")
    return out


def gpu_baseline(scene, w, h, calls=6):
    """The reference's own GPU megakernel on this GPU (speed only)."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import refdrv
    import tinsel_b200 as tb
    if not (refdrv.have_ref_gpu() and refdrv.have_ref("literal")):
        return None
    sc = refdrv.RefScene.from_snapshot(tb.scene_path(scene), "literal")
    sc.set_size(w, h)
    try:
        wall_ms, kern_ms = sc.gpu_bench(2, calls)
    finally:
        sc.close()
    n = w * h
    return {"impl": "tinsel src/render.cu RenderGpu (reference GPU megakernel, its Release flags, sm_100a)",
            "value": n / kern_ms / 1e3, "e2e": n / wall_ms / 1e3, "unit": "Msamples/s",
            "kernel_ms_per_spp": kern_ms, "render_call_ms": wall_ms,
            "note": "a different, fast-math estimator (SURVEY 2 row 3): speed bar only, not a parity arm"}


def dump_outputs(np, outdir, accum):
    """Writes what the timed path hands its caller after the last timed step: the accumulator, (H, W, 4)
    float32 running sums (sum w*rgb, sum w) over every timed sample.  r.Init resets the frame index, so
    the same --steps give the same samples whatever --warmup is."""
    os.makedirs(outdir, exist_ok=True)
    np.save(os.path.join(outdir, "accumulator.npy"), np.ascontiguousarray(accum, np.float32))


def measure_one_gpu(tb, torch, np, scene, w, h, spp, steps, warmup, device, flush, want_clocks=False, dump=None):
    """Single-GPU measurement of one configuration: device-resident value + e2e through tb200_render.
    dump: directory for the timed path's output (dump_outputs)."""
    snap = tb.Snapshot(tb.scene_path(scene))
    cam, opt = snap.camera, snap.options
    opt.width, opt.height = w, h
    r = tb.Renderer(snap.scene, device=device)
    r.Init(w, h)
    stream = torch.cuda.Stream()
    with torch.cuda.stream(stream):
        r.set_stream(stream.cuda_stream)
        for _ in range(warmup):
            r.render_device(cam, opt, spp)
        r.Init(w, h)
        torch.cuda.synchronize()
        clocks = ClockSampler(device) if want_clocks else None
        if clocks:
            clocks.start()
        launches0 = r.stats().kernelLaunches
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        lib_ms = []
        for i in range(steps):
            flush.fill_(i & 0xff)                       # evict L2 between timed steps (same stream, not timed)
            ev[i][0].record(stream)
            r.render_device(cam, opt, spp)              # synchronous: returns when the step's kernels are done
            ev[i][1].record(stream)
            lib_ms.append(r.stats().gpuMs)              # the library's own CUDA events around the launch, same stream
        torch.cuda.synchronize()
        if clocks:
            clocks.stop_flag = True
            clocks.join(timeout=2)
        # Two event pairs bracket every step on the launching stream: torch's, recorded from Python around the call,
        # and the library's, recorded in C right around the launch.  The first also counts the host's delay between
        # recording the event and launching the kernel (tens of microseconds; milliseconds when eight ranks share a
        # CPU quota), so the step time is the library's and torch's is reported next to it.
        torch_ms = [a.elapsed_time(b) for a, b in ev]
        step_ms = lib_ms
        launches = r.stats().kernelLaunches - launches0
        img = r.read_accumulator()
    if dump:
        dump_outputs(np, dump, img)
    value = w * h * spp * steps / sum(step_ms) / 1e3

    # sanity: filter weights sum to spp per interior pixel
    xs = (np.arange(4000) + 0.5) / 4000.0 * 2.0 - 1.0
    fw = opt.filterWidth
    g = np.maximum(0.0, np.exp(-opt.filterFalloff * (xs * fw) ** 2) - opt.filterOffset)
    expect = float((g.sum() * (2.0 * fw / 4000.0)) ** 2) * spp * steps
    wsum = float(img[4:-4, 4:-4, 3].mean())
    assert abs(wsum / expect - 1.0) < 0.01, (scene, wsum, expect)
    assert np.isfinite(img).all() and float(img[..., :3].sum()) > 0.0

    # e2e: Renderer::Render through the C ABI, HOST output buffer (pinned by the caller, who owns it)
    r.set_stream(None)
    r.Init(w, h)
    host = np.zeros((h, w, 4), np.float32)
    r.pin_output(host)
    for _ in range(3):
        r.Render(cam, opt, host)
    calls = E2E_CALLS_PER_STEP * steps
    t0 = time.time()
    for _ in range(calls):
        r.Render(cam, opt, host)
    e2e_dt = time.time() - t0
    assert abs(float(host[4:-4, 4:-4, 3].mean()) / (expect / (spp * steps) * (calls + 3)) - 1.0) < 0.01
    r.close()
    snap.close()
    res = {"value": value, "step_ms": step_ms, "torch_event_ms": torch_ms, "launches": launches,
           "e2e_value": w * h * calls / e2e_dt / 1e6, "e2e_ms_per_call": e2e_dt / calls * 1e3, "e2e_calls": calls,
           "cam_opt_bytes": C.sizeof(tb.Camera) + C.sizeof(tb.Options)}
    if clocks:
        res["clocks"] = clocks.summary()
    return res


def run_ours(args):
    import numpy as np
    import torch
    import tinsel_b200 as tb

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the product path has no CPU fallback)")
    torch.cuda.set_device(local)
    os.environ.pop("TINSEL_B200_PIPELINE", None)
    scene, W, H, SPP = MAIN
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    if world == 1:
        res = measure_one_gpu(tb, torch, np, scene, W, H, SPP, args.steps, args.warmup, local, flush, want_clocks=True,
                              dump=args.dump_outputs)
        value, step_ms = res["value"], res["step_ms"]
        avg_launch_s = sum(step_ms) / len(step_ms) / 1e3
        line = {
            "metric": "Msamples/sec (paths x spp / s)", "value": value, "unit": "Msamples/s",
            "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": sum(step_ms) / args.steps, "ms_per_step_torch_events": sum(res["torch_event_ms"]) / args.steps,
            "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic (scene snapshot, random paths)",
            "config": workload_config(scene, W, H, SPP, 1),
            "clocks": res["clocks"],
            "e2e": {"value": res["e2e_value"], "unit": "Msamples/s",
                    "h2d_bytes_per_step": E2E_CALLS_PER_STEP * res["cam_opt_bytes"],
                    "d2h_bytes_per_step": E2E_CALLS_PER_STEP * W * H * 16,
                    "calls_per_step": E2E_CALLS_PER_STEP, "ms_per_call": res["e2e_ms_per_call"]},
            "gpu_launches": res["launches"],
            "roofline": roofline_block(scene, value, avg_launch_s, W * H * SPP, res["clocks"].get("sm_mhz")),
        }
        try:
            gb = gpu_baseline(scene, W, H)
        except Exception as e:  # noqa: BLE001 -- a secondary arm must not cost the headline line
            gb = {"unavailable": str(e)}
        if gb:
            line["gpu_baseline"] = gb
        # the other BASELINE.json GPU configurations, same measurements, fewer steps
        if not args.no_configs:
            configs = {}
            for name, (w, h, spp) in OTHER_WORKLOADS.items():
                if not os.path.exists(tb.scene_path(name)):
                    configs[name] = {"unavailable": "scenes/%s.tsnap is not on this box" % name}
                    continue
                try:
                    # 4 warm-up launches: the split-queue tuner (api.cu tune_update) has decided by then
                    sub = measure_one_gpu(tb, torch, np, name, w, h, spp, 3, 4, local, flush)
                    sub_gb = gpu_baseline(name, w, h, 3)
                except Exception as e:  # noqa: BLE001
                    configs[name] = {"error": str(e)}
                    continue
                sms = sub["step_ms"]
                configs[name] = {
                    "workload": "data/%s.tin %dx%d, %d spp per step" % (name, w, h, spp),
                    "value": sub["value"], "ms_per_step": sum(sms) / len(sms),
                    "e2e": {"value": sub["e2e_value"], "ms_per_call": sub["e2e_ms_per_call"], "d2h_bytes_per_call": w * h * 16},
                    "roofline": roofline_block(name, sub["value"], sum(sms) / len(sms) / 1e3, w * h * spp, res["clocks"].get("sm_mhz")),
                    "gpu_baseline": sub_gb,
                }
            line["configs"] = configs
        arm = CpuArm(scene, W, H)
        arm.warm()
        cpu_msps, cpu_dt = arm.timed(16)
        line["cpu_baseline"] = {"value": cpu_msps, "unit": "Msamples/s", "cores": arm.threads, "kind": arm.kind,
                                "sample": "%dx%d image, 16 spp (%.1f s wall), per-sample-seeded work-stealing driver over the "
                                          "reference's PathTrace/AddSample, after a 1.5 s warm-up of the host cores" % (W, H, cpu_dt)}
        arm.close()
        print(json.dumps(line), flush=True)
        return

    # ---------------------------------- N > 1: one rank per GPU -----------------------------------
    import torch.distributed as dist
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    host_group = dist.new_group(backend="gloo")     # host-side barriers: waiting ranks must not occupy their GPU

    snap = tb.Snapshot(tb.scene_path(scene))
    cam, opt = snap.camera, snap.options
    opt.width, opt.height = W, H
    r = tb.Renderer(snap.scene, device=local)
    r.Init(W, H)
    r.set_shard(rank, world)
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    accum = torch.zeros((H, W, 4), dtype=torch.float32, device="cuda")
    r.bind_accumulator(accum.data_ptr())
    r.set_stream(stream.cuda_stream)

    def barrier():
        dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        r.render_device(cam, opt, SPP)
    dist.reduce(accum.clone(), dst=0)   # warm the communicator
    accum.zero_()
    r.set_frame(0)
    barrier()

    clocks = ClockSampler(local)
    clocks.start()
    launches0 = r.stats().kernelLaunches
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps + 1)]
    lib_ms = []
    for i in range(args.steps):
        flush.fill_(i & 0xff)
        ev[i][0].record(stream)
        r.render_device(cam, opt, SPP)
        ev[i][1].record(stream)
        lib_ms.append(r.stats().gpuMs)
    # the reduce is timed from a common start: without the barrier, its events on the early ranks would also
    # count the time they wait for a rank whose host thread was descheduled between two steps (4 ms seen at N = 8)
    barrier()
    ev[args.steps][0].record(stream)
    dist.reduce(accum, dst=0, op=dist.ReduceOp.SUM)
    ev[args.steps][1].record(stream)
    barrier()
    clocks.stop_flag = True
    clocks.join(timeout=2)
    torch_ms = [a.elapsed_time(b) for a, b in ev[:args.steps]]
    step_ms = lib_ms       # the library's events around the launch (see measure_one_gpu)
    reduce_ms = ev[args.steps][0].elapsed_time(ev[args.steps][1])
    dev_ms = sum(step_ms) + reduce_ms
    launches = r.stats().kernelLaunches - launches0
    t = torch.tensor([dev_ms, float(launches)], dtype=torch.float64, device="cuda")
    tmax = t.clone()
    dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    tsum = t.clone()
    dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
    dev_ms = float(tmax[0])
    launches = int(tsum[1])
    value = W * H * SPP * args.steps / dev_ms / 1e3
    # every rank's clocks and its own device time: on a shared 8-GPU box single GPUs have been seen 25-35 % slower
    # than their neighbours under full load, and the max over ranks is what `value` reports
    per_rank = [None] * world
    dist.all_gather_object(per_rank, {"rank": rank, "steps_ms": round(sum(step_ms), 3), "steps_ms_torch_events": round(sum(torch_ms), 3),
                                      "clocks": clocks.summary()}, group=host_group)
    if rank == 0:
        img = accum.cpu().numpy()
        assert np.isfinite(img).all() and float(img[..., :3].sum()) > 0.0
        if args.dump_outputs:
            dump_outputs(np, args.dump_outputs, img)
    r.close()
    del accum
    torch.cuda.synchronize()
    dist.barrier(group=host_group)

    # ---- e2e: the product's own multi-GPU path, one renderer over all N devices, driven by rank 0 --
    e2e = None
    if rank == 0:
        m = tb.Renderer(snap.scene, devices=list(range(world)))
        m.Init(W, H)
        host = np.zeros((H, W, 4), np.float32)
        m.pin_output(host)
        for _ in range(3):
            m.Render(cam, opt, host)
        calls = E2E_CALLS_PER_STEP * args.steps
        t0 = time.time()
        for _ in range(calls):
            m.Render(cam, opt, host)
        e2e_dt = time.time() - t0
        assert np.isfinite(host).all() and float(host[..., 3].min()) > 0.0   # every row was delivered by its owner
        per_device = []
        for k in range(world):
            st, row0, rows = m.member_stats(k)
            per_device.append({"device": k, "rows": [row0, row0 + rows], "kernel_ms_last_call": round(st.gpuMs, 4)})
        e2e = {"value": W * H * calls / e2e_dt / 1e6, "unit": "Msamples/s", "per_device": per_device,
               "h2d_bytes_per_step": E2E_CALLS_PER_STEP * (C.sizeof(tb.Camera) + C.sizeof(tb.Options)),
               "d2h_bytes_per_step": E2E_CALLS_PER_STEP * W * H * 16,
               "calls_per_step": E2E_CALLS_PER_STEP, "ms_per_call": e2e_dt / calls * 1e3,
               "path": "tb200_create_multi over %d devices: row slabs, per-device streamed read-back, no reduce" % world}
        m.close()
    dist.barrier(group=host_group)

    if rank == 0:
        per_launch_samples = W * H * SPP / world
        avg_launch_s = (sum(step_ms) / len(step_ms)) / 1e3
        line = {
            "metric": "Msamples/sec (paths x spp / s)", "value": value, "unit": "Msamples/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic (scene snapshot, random paths)",
            "config": workload_config(scene, W, H, SPP, world),
            "clocks": dict(clocks.summary(), per_rank=per_rank),
            "e2e": e2e,
            "gpu_launches": launches,
            "roofline": roofline_block(scene, value / world, avg_launch_s, per_launch_samples, clocks.summary().get("sm_mhz")),
            "reduce_ms": reduce_ms,
        }
        arm = CpuArm(scene, W, H)
        arm.warm()
        cpu_msps, cpu_dt = arm.timed(16)
        line["cpu_baseline"] = {"value": cpu_msps, "unit": "Msamples/s", "cores": arm.threads, "kind": arm.kind,
                                "sample": "%dx%d image, 16 spp (%.1f s wall), work-stealing driver over the reference's PathTrace" % (W, H, cpu_dt)}
        arm.close()
        print(json.dumps(line), flush=True)
    snap.close()
    dist.barrier(group=host_group)
    dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--scene", default="cornell", choices=["cornell"] + sorted(OTHER_WORKLOADS),
                    help="run another BASELINE.json configuration as the main workload (development)")
    ap.add_argument("--no-configs", action="store_true", help="skip the sub-results for the other BASELINE.json configurations")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the timed path's output after the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the GPU path's output: use it with --impl ours")
    if args.scene != "cornell":
        global MAIN
        w, h, spp = OTHER_WORKLOADS[args.scene]
        MAIN = (args.scene, w, h, spp)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
