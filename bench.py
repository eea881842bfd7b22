#!/usr/bin/env python3
"""Benchmark of the hot path at 7680x4320 (BASELINE.json: "frames/sec encode (UYVY->DXT1, UYVY->JPEG); HBM GB/s vs roofline").

  python bench.py --gpus N --steps K --warmup W            (N>1: launched by torch.distributed.run, one rank per GPU)
  python bench.py --impl reference ...                      CPU arm (rank 0 only; see reference_arm)

Headline (the top-level keys of the JSON line) = fused UYVY -> DXT1.  A "step" = P passes over a batch of B distinct 8K frames
resident in HBM (B x 66 MB is far larger than the 126 MB L2, nothing is served from cache); the B launches of a pass are captured
in a CUDA graph in the order of the frame indices this rank received, a step replays it P times.  Frames are independent units:
with N GPUs each rank encodes its own batch (weak scaling, no data-path collective); the only collective is the NCCL scatter of
the int32 frame indices, one step ahead on a side stream, and the encode order is built from (and every step checked against)
what arrived.

`workloads` carries the other BASELINE configs in the same shape (value / roofline / e2e / cpu_baseline), at every N:
  uyvy_jpeg_8k_q90     second half of the metric      rgb_jpeg_8k_q90   config 3 (three scans)
  uyvy_dxt5ycocg_8k    config 5 (one stream per GPU)  v210_p010_8k      config 4
`e2e` numbers go through the reference-facing plugin (compress_init / compress_frame / compress_pop, or the C ABI for the planar
converter) with pinned HOST frames: H2D + kernels + D2H inside the timed region, every frame.
"""
import argparse
import json
import os
import sys
import threading
import time

LAUNCH_AFFINITY = os.sched_getaffinity(0)  # before anything loads libgomp: with OMP_PROC_BIND its initialisation pins the calling thread
if "--impl" in sys.argv and "reference" in sys.argv:  # CPU arm only: OpenMP threads stay where they start (must be set before libgomp loads;
    os.environ.setdefault("OMP_PROC_BIND", "close")   # the GPU arm leaves torch's OpenMP runtime alone)
    os.environ.setdefault("OMP_PLACES", "cores")

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

W8K, H8K = 7680, 4320
PX = W8K * H8K
UYVY, V210, RGB = 2, 7, 12
ALGO = {  # algorithmic bytes per frame, SURVEY.md section 8(d): compulsory input read + output write
    "uyvy_dxt1": PX * 2 + PX // 2,           # 2 + 0.5 B/px
    "uyvy_dxt5": PX * 2 + PX,                # 2 + 1
    "v210_p010": PX * 16 // 6 + PX * 3,      # 16/6 + 3
}
METRIC = "7680x4320 frames/sec encode (UYVY->DXT1)"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--frames", type=int, default=48, help="distinct 8K frames per pass per GPU")
    ap.add_argument("--passes", type=int, default=16, help="passes over the batch per step (timed region >= 0.5 s at the default K)")
    ap.add_argument("--no-extra", action="store_true", help="headline only (profiling runs)")
    ap.add_argument("--only", default="", help="comma-separated subset of the secondary workloads")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the headline encode produced in the last one "
                    "(a fixed sample of the DXT1 blocks of every frame of rank 0) to DIR/*.npy")
    return ap.parse_args()


DUMP_BYTES = 48 << 20  # the dump stays well below 64 MB whatever the batch size


def dump_dxt1(outs, out_dir):
    """DIR/dxt1_blocks.npy: float64 (frames, blocks, 2), the two 32-bit words (colours, indices) of the same seeded sample of block
    positions in every frame; DIR/dxt1_block_index.npy: those positions (row-major 4x4 blocks).  The integers are exact in float64."""
    import numpy as np
    import torch
    n_frames, n_blocks = outs.shape[0], outs.shape[1] // 8
    n = min(n_blocks, DUMP_BYTES // (16 * n_frames + 8))  # 16 bytes per block and frame, 8 per position
    idx = np.sort(np.random.default_rng(0).choice(n_blocks, size=n, replace=False))
    words = outs.view(torch.int32).reshape(n_frames, n_blocks, 2)[:, torch.from_numpy(idx).to(outs.device)]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "dxt1_blocks.npy"), (words.cpu().numpy().astype(np.int64) & 0xFFFFFFFF).astype(np.float64))
    np.save(os.path.join(out_dir, "dxt1_block_index.npy"), idx.astype(np.float64))


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def traffic_of(key):
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            return json.load(f).get(key)
    except Exception:
        return None


def effective_cpus():
    """CPUs this process may really use: affinity mask at launch capped by the cgroup quota (cpu.max) — OpenMP's own view ignores the quota
    (round 1: 128 threads on a 16-CPU quota ran the port at a sixth of its speed)"""
    aff = len(LAUNCH_AFFINITY)
    quota = None
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            with open(path) as f:
                parts = f.read().split()
            if path.endswith("cpu.max"):
                if parts[0] != "max":
                    quota = float(parts[0]) / float(parts[1])
            else:
                q = float(parts[0])
                if q > 0:
                    with open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as f:
                        quota = q / float(f.read())
            break
        except Exception:
            continue
    eff = aff if quota is None else max(1, min(aff, int(quota + 0.5)))
    return {"affinity": aff, "cgroup_quota": quota, "used": eff, "os_cpu_count": os.cpu_count()}


class ClockSampler:
    """SM clock + throttle reasons sampled through NVML while the timed region runs"""

    def __init__(self, uuid=None, index=0):
        self.uuid, self.index, self.rows, self.stop_flag, self.thread = uuid, index, [], False, None
        self.max_mhz, self.t0, self.t1 = None, None, None

    def _run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = None
            if self.uuid:
                for cand in (f"GPU-{self.uuid}", str(self.uuid)):
                    try:
                        h = nv.nvmlDeviceGetHandleByUUID(cand.encode() if isinstance(cand, str) else cand)
                        break
                    except Exception:
                        h = None
            if h is None:
                h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            while not self.stop_flag:
                try:
                    reasons = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:
                    reasons = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                self.rows.append((nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM), reasons, time.perf_counter()))
                time.sleep(0.002)
        except Exception as e:  # noqa: BLE001
            self.rows.append(("error", str(e)))

    def start(self):
        self.thread = threading.Thread(target=self._run, daemon=True)
        self.thread.start()

    def window_begin(self):
        self.t0 = time.perf_counter()

    def window_end(self):
        self.t1 = time.perf_counter()

    def stop(self):
        self.stop_flag = True
        if self.thread:
            self.thread.join(timeout=2)
        good = [r for r in self.rows if r[0] != "error" and (self.t0 is None or self.t0 <= r[2] <= (self.t1 or 1e30))]
        sm = sorted(r[0] for r in good)
        names = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}
        reasons = sorted({n for r in good for bit, n in names.items() if r[1] & bit})
        err = [r[1] for r in self.rows if r[0] == "error"]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.max_mhz, "reasons": reasons, "samples": len(sm),
                **({"error": err[0]} if err else {})}


# =====================================================================================================================
# CPU side: the oracle port / the reference objects on the host cores (cpu_baseline, --impl reference)
# =====================================================================================================================
def _natural_uyvy_cpu(orc, seed=1):
    import numpy as np
    import util
    yy, xx = np.mgrid[0:H8K, 0:W8K]
    rgb = np.stack([xx * 255 // (W8K - 1), yy * 255 // (H8K - 1), (xx + yy) % 256], axis=2).astype(np.int16)
    rgb = (rgb + np.random.default_rng(seed).integers(-6, 7, rgb.shape, dtype=np.int16)).clip(0, 255).astype(np.uint8)
    return util.convert_cpu(orc, "orc_convert", RGB, UYVY, rgb.reshape(-1), W8K, H8K), rgb.reshape(-1)


def cpu_workload(name, orc, ref, frames=None):
    """returns (callable encoding ONE 8K frame on all usable host threads, kind, description)"""
    import ctypes
    import numpy as np
    import util
    if name == "uyvy_dxt1":
        src = util.rng_bytes(PX * 2, 4)
        out = np.zeros(PX // 2, dtype=np.uint8)
        return (lambda: orc.orc_uyvy_to_dxt1(src.ctypes.data, out.ctypes.data, W8K, H8K, 0)), "port", \
            "oracle/dxt_oracle.c (cuda_dxt's arithmetic; UltraGrid has no CPU DXT encoder), OpenMP over block rows, noise frame"
    if name == "uyvy_dxt5":
        src = util.rng_bytes(PX * 2, 4)
        out = np.zeros(PX, dtype=np.uint8)
        fn = getattr(orc, "orc_uyvy_to_dxt6", None)
        if fn is None:
            return None, "port", "no CPU port of the fused DXT5 path"
        return (lambda: fn(src.ctypes.data, out.ctypes.data, W8K, H8K, 0)), "port", "oracle/dxt_oracle.c DXT5-YCoCg, OpenMP over block rows, noise frame"
    if name in ("uyvy_jpeg", "rgb_jpeg"):
        uyvy, rgb = frames if frames is not None else _natural_uyvy_cpu(orc)
        src = uyvy if name == "uyvy_jpeg" else rgb
        fmt = 0 if name == "uyvy_jpeg" else 1
        cap = PX * 3 // 64 * 418 + 4096 if fmt else PX * 2 // 64 * 418 + 4096
        out = np.zeros(cap, dtype=np.uint8)
        orc.orc_jpeg_encode_parallel.restype = ctypes.c_size_t
        orc.orc_jpeg_encode_parallel.argtypes = [ctypes.c_void_p, ctypes.c_long, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                                 ctypes.c_void_p, ctypes.c_size_t]
        return (lambda: orc.orc_jpeg_encode_parallel(src.ctypes.data, W8K * (3 if fmt else 2), W8K, H8K, fmt, 90, 0, out.ctypes.data, out.size)), "port", \
            "oracle/jpeg_oracle.c orc_jpeg_encode_parallel (GPUJPEG is not in the tree), OpenMP over restart segments, natural frame q=90"
    if name == "v210_p010":
        src = util.v210_noise(W8K, H8K, 3)
        # the chroma buffer is a whole frame: decode_to_planar_parallel offsets EVERY plane of band i by i * rows * linesize (to_planar.c:511-515),
        # also the half-height CbCr plane, so the upper bands land beyond a tight plane
        y, c = np.zeros(PX * 2, np.uint8), np.zeros(PX * 2, np.uint8)
        if ref is not None:
            return (lambda: ref.ref_v210_to_p010le_parallel(W8K, H8K, y.ctypes.data, W8K * 2, c.ctypes.data, W8K * 2, src.ctypes.data, 0)), "reference", \
                "UNMODIFIED src/to_planar.c decode_to_planar_parallel(v210_to_p010le, TO_PLANAR_THREADS_AUTO) from oracle/_ref (-O3 -msse4.1)"
        return (lambda: orc.orc_v210_to_p010le(W8K, H8K, y.ctypes.data, W8K * 2, c.ctypes.data, W8K * 2, src.ctypes.data)), "port", "oracle/planar_oracle.c, 1 thread"
    raise KeyError(name)


def time_cpu(fn, budget_s=8.0, min_runs=5, max_runs=12):
    """wall time per call: best and median of >= 5 runs (one warm-up first), bounded by a time budget"""
    fn()
    times, t_all = [], time.perf_counter()
    while len(times) < min_runs or (len(times) < max_runs and time.perf_counter() - t_all < budget_s):
        t0 = time.perf_counter()
        fn()
        times.append(time.perf_counter() - t0)
        if time.perf_counter() - t_all > 4 * budget_s:
            break
    times.sort()
    return times[0], times[len(times) // 2], len(times)


def cpu_baseline_block(name, orc, ref, cpus, frames=None, budget_s=8.0):
    fn, kind, what = cpu_workload(name, orc, ref, frames)
    if fn is None:
        return {"value": None, "unit": "frames/s", "cores": cpus["used"], "kind": kind, "sample": what}
    best, med, n = time_cpu(fn, budget_s)
    return {"value": 1.0 / med, "unit": "frames/s", "cores": cpus["used"], "kind": kind, "best": 1.0 / best,
            "sample": f"median of {n} single 7680x4320 frames ({med * 1e3:.1f} ms; best {best * 1e3:.1f} ms): {what}", "cpus": cpus}


def reference_arm(args, rank):
    """CPU arm.  The reference has no CPU implementation of DXT or JPEG encode (DXT: CUDA / GLSL only; JPEG: libgpujpeg), so for those the arm
    is the oracle port of the same arithmetic on every usable host thread (kind "port"); for v210->P010 it is the reference's own objects
    (kind "reference").  One step = one 8K frame (a bounded sample of the GPU arm's batch).  Rank 0 alone works."""
    if rank != 0:
        return
    import util
    cpus = effective_cpus()  # before libgomp loads: OMP_PROC_BIND pins the calling thread to one place and the mask would read 1
    orc, ref = util.oracle(), util.ref_cpu()
    orc.orc_set_threads(cpus["used"])
    fn, kind, what = cpu_workload("uyvy_dxt1", orc, ref)
    for _ in range(max(args.warmup, 1)):
        fn()
    times = []
    for _ in range(args.steps):
        t0 = time.perf_counter()
        fn()
        times.append(time.perf_counter() - t0)
    dt = sum(times)
    fps = args.steps / dt
    st = sorted(times)
    line = {
        "impl": "reference", "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "7680x4320 UYVY->DXT1 encode on host cores, 1 noise frame per step", "note": what},
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": cpus["used"], "kind": kind, "best": 1.0 / st[0], "median": 1.0 / st[len(st) // 2],
                         "sample": f"{args.steps} noise frames 7680x4320, one per step", "cpus": cpus,
                         "omp": {k: os.environ.get(k) for k in ("OMP_NUM_THREADS", "OMP_PROC_BIND", "OMP_PLACES")}},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    if not args.no_extra:
        wl, frames = {}, None
        for name in ("uyvy_jpeg", "rgb_jpeg", "uyvy_dxt5", "v210_p010"):
            try:
                if name.endswith("jpeg") and frames is None:
                    frames = _natural_uyvy_cpu(orc)
                b = cpu_baseline_block(name, orc, ref, cpus, frames, budget_s=5.0)
                wl[name] = {"impl": "reference", "value": b["value"], "unit": "frames/s", "cpu_baseline": b,
                            "e2e": {"value": b["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
            except Exception as e:  # noqa: BLE001
                wl[name] = {"error": f"{type(e).__name__}: {e}"[:200]}
        line["workloads"] = wl
    print(json.dumps(line))


# =====================================================================================================================
# GPU side
# =====================================================================================================================
class Ctx:
    pass


def dev_timed(ctx, fn, iters, warm=3):
    """CUDA-event time of `iters` calls of fn(i) on the current stream, max over ranks, seconds per call"""
    torch = ctx.torch
    for i in range(warm):
        fn(i)
    ctx.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(iters):
        fn(i)
    e1.record()
    ctx.barrier()
    return ctx.max_over_ranks(e0.elapsed_time(e1) * 1e-3) / iters


def graph_timed(ctx, fn, launches, replays, warm=2):
    """`launches` calls of fn(i) captured into one CUDA graph, replayed `replays` times between two events: per-launch seconds (max over
    ranks).  The Python / ctypes cost of a launcher is outside the timed region."""
    torch = ctx.torch
    for i in range(min(launches, 4)):
        fn(i)
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.stream(s):
        with torch.cuda.graph(g, stream=s, capture_error_mode="thread_local"):  # NCCL's watchdog thread polls events meanwhile
            for i in range(launches):
                fn(i)
        for _ in range(warm):
            g.replay()
        s.synchronize()
        ctx.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(s)
        for _ in range(replays):
            g.replay()
        e1.record(s)
        s.synchronize()
    ctx.barrier()
    return ctx.max_over_ranks(e0.elapsed_time(e1) * 1e-3) / (launches * replays)


def roofline(ctx, algo_bytes, secs, kernel, traffic_key=None, **more):
    ach = algo_bytes / secs / 1e9
    return {"bound": "hbm", "achieved": ach, "peak": ctx.peak, "unit": "GB/s", "frac": ach / ctx.peak, "traffic": traffic_of(traffic_key) if traffic_key else None,
            "kernel": kernel, "algorithmic_bytes_per_launch": algo_bytes, "us_per_launch": secs * 1e6, "peak_source": ctx.peak_src, **more}


def module_e2e(ctx, cfg, hosts, w, h, codec, frames, depth, out_check=None):
    """frames through compress_init(cfg) / compress_frame / compress_pop with pinned host input, `depth` in flight, results popped in order
    (zero-copy view of the pooled pinned output frame).  Wall clock between two device synchronisations, max over ranks -> frames/s of all ranks"""
    torch, compress = ctx.torch, ctx.compress
    c = compress.Compress(cfg)

    def run(n):
        inflight, last = 0, None
        for i in range(n):
            c.push(hosts[i % len(hosts)], w, h, codec)
            inflight += 1
            if inflight == depth:
                last = c.pop_ref()[0]
                inflight -= 1
        while inflight:
            last = c.pop_ref()[0]
            inflight -= 1
        return last
    last = run(2 * depth + 2)  # lanes have their buffers, the pool its pinned frames
    if out_check is not None:
        out_check(last)
    ctx.barrier()
    t0 = time.perf_counter()
    run(frames)
    torch.cuda.synchronize()
    dt = ctx.max_over_ranks(time.perf_counter() - t0)
    c.close()
    return ctx.world * frames / dt


def host_copy(ctx, t):
    """device tensor -> pinned host numpy array on the GPU's NUMA node"""
    a = ctx.api.pinned_near(t.numel(), ctx.local_rank)
    ctx.torch.from_numpy(a).copy_(t)
    return a


def wl_dxt5(ctx, frames):
    """config 5: UYVY -> DXT5-YCoCg, one stream (batch of frames) per GPU"""
    torch, api = ctx.torch, ctx.api
    B = min(len(frames), 12)
    outs = [torch.empty(PX, dtype=torch.uint8, device=ctx.dev) for _ in range(2)]
    secs = graph_timed(ctx, lambda i: api.uyvy_to_dxt(frames[i % B], W8K, H8K, dxt_type=6, out=outs[i & 1]), B, max(4, int(0.4 / (B * 90e-6))))
    hosts = [host_copy(ctx, frames[i]) for i in range(4)]
    e2e = module_e2e(ctx, "cuda_dxt:DXT5", hosts, W8K, H8K, UYVY, 200, 3)
    return {"metric": "7680x4320 frames/sec encode (UYVY->DXT5-YCoCg)", "value": ctx.world / secs, "unit": "frames/s", "ms_per_frame": secs * 1e3,
            "config": {"workload": "BASELINE config 5: 8K UYVY->DXT5-YCoCg fused encode, one stream of noise frames per GPU", "frames": B},
            "roofline": roofline(ctx, ALGO["uyvy_dxt5"], secs, "ugb::dxt_uyvy_kernel<6,1,false>", "dxt6_uyvy_kernel_8k_bytes_per_launch"),
            "e2e": {"value": e2e, "unit": "frames/s", "h2d_bytes_per_frame": PX * 2, "d2h_bytes_per_frame": PX,
                    "path": "compress_init('cuda_dxt:DXT5'), pinned host UYVY in, pooled pinned DXT5 out, 3 frames in flight"},
            "gpu_launches_per_frame": 1}


def wl_p010(ctx):
    """config 4: v210 -> P010 (4:2:0 semi-planar 10-bit in 16), HBM-bandwidth workload"""
    torch, api = ctx.torch, ctx.api
    from ultragrid_b200 import Codec, vc_get_linesize
    ls = vc_get_linesize(W8K, Codec.v210)
    nb = 6
    g = torch.Generator(device=ctx.dev)
    g.manual_seed(77 + ctx.rank)
    src = [torch.randint(0, 1 << 30, (ls // 4 * H8K,), dtype=torch.int32, device=ctx.dev, generator=g).view(torch.uint8) for _ in range(nb)]
    oy = [torch.empty(PX * 2, dtype=torch.uint8, device=ctx.dev) for _ in range(2)]
    oc = [torch.empty(PX, dtype=torch.uint8, device=ctx.dev) for _ in range(2)]
    secs = graph_timed(ctx, lambda i: api.v210_to_p010le(src[i % nb], W8K, H8K, out_y=oy[i & 1], out_c=oc[i & 1]), nb, max(4, int(0.4 / (nb * 36e-6))))
    # end to end through the C ABI with host buffers: 3 slots, each H2D -> kernel -> D2H (two planes) on its own stream
    slots = []
    for k in range(3):
        slots.append({"st": torch.cuda.Stream(), "hin": torch.from_numpy(host_copy(ctx, src[k])), "din": torch.empty_like(src[0]),
                      "dy": torch.empty(PX * 2, dtype=torch.uint8, device=ctx.dev), "dc": torch.empty(PX, dtype=torch.uint8, device=ctx.dev),
                      "hy": torch.from_numpy(api.pinned_near(PX * 2, ctx.local_rank)), "hc": torch.from_numpy(api.pinned_near(PX, ctx.local_rank))})

    def run(n):
        for i in range(n):
            s = slots[i % 3]
            s["st"].synchronize()  # the slot's previous frame is on the host
            with torch.cuda.stream(s["st"]):
                s["din"].copy_(s["hin"], non_blocking=True)
                api.v210_to_p010le(s["din"], W8K, H8K, out_y=s["dy"], out_c=s["dc"], stream=s["st"])
                s["hy"].copy_(s["dy"], non_blocking=True)
                s["hc"].copy_(s["dc"], non_blocking=True)
        for s in slots:
            s["st"].synchronize()
    run(6)
    ctx.barrier()
    n = 150
    t0 = time.perf_counter()
    run(n)
    dt = ctx.max_over_ranks(time.perf_counter() - t0)
    del slots
    return {"metric": "7680x4320 frames/sec convert (v210->P010)", "value": ctx.world / secs, "unit": "frames/s", "ms_per_frame": secs * 1e3,
            "config": {"workload": "BASELINE config 4: 8K v210->P010 (v210_to_p010le), 30-bit noise frames", "frames": nb},
            "roofline": roofline(ctx, ALGO["v210_p010"], secs, "ugb::v210_to_p010_kernel<4>", "v210_to_p010_kernel_8k_bytes_per_launch"),
            "e2e": {"value": ctx.world * n / dt, "unit": "frames/s", "h2d_bytes_per_frame": ls * H8K, "d2h_bytes_per_frame": PX * 3,
                    "path": "ugb200_v210_to_p010le through the C ABI: pinned host v210 -> H2D -> kernel -> D2H of both planes, 3 slots on 3 streams"},
            "gpu_launches_per_frame": 1}


def natural_frames(ctx, n):
    """ramps + noise RGB frames made on the device and their UYVY form through the product's own (reference-exact) RGB->UYVY converter"""
    torch, api = ctx.torch, ctx.api
    xx = torch.arange(W8K, device=ctx.dev, dtype=torch.int32).view(1, W8K)
    yy = torch.arange(H8K, device=ctx.dev, dtype=torch.int32).view(H8K, 1)
    base = torch.stack([(xx * 255 // (W8K - 1)).expand(H8K, W8K), (yy * 255 // (H8K - 1)).expand(H8K, W8K), (xx + yy) % 256], dim=2)
    g = torch.Generator(device=ctx.dev)
    rgbs, uyvys = [], []
    for k in range(n):
        g.manual_seed(1000 * ctx.rank + k)
        rgb = (base + torch.randint(-6, 7, base.shape, dtype=torch.int32, device=ctx.dev, generator=g)).clamp_(0, 255).to(torch.uint8).reshape(-1)
        rgbs.append(rgb)
        uyvys.append(api.pixfmt_convert(RGB, UYVY, rgb, W8K, H8K))
    del base
    return rgbs, uyvys


def wl_jpeg(ctx, name, codec, frames, cfg_note):
    """UYVY -> JPEG (second half of the metric) / RGB -> JPEG (config 3), q = 90, GPUJPEG's stream layout for that input (gpujpeg.cpp:295-305)"""
    torch, api = ctx.torch, ctx.api
    bpp = 2 if codec == UYVY else 3
    enc = api.JpegEncoder()
    sizes = []
    for f in frames:  # the encoder sizes its bit buffers (and with them the kernel instantiation) from the previous frame's statistics
        for _ in range(2):
            enc.encode_device(f, W8K, H8K, codec, quality=90)
            nbytes = enc.result_size()
        sizes.append(nbytes)
    nf = len(frames)
    stream_bytes = sum(sizes) / nf
    per = dev_timed(ctx, lambda i: enc.encode_device(frames[i % nf], W8K, H8K, codec, quality=90), max(24, int(0.35 / 180e-6)), warm=4)
    enc.result_size()
    enc.stage_timing(True)
    st = [0.0, 0.0, 0.0, 0.0]
    for i in range(nf):
        enc.encode_device(frames[i], W8K, H8K, codec, quality=90)
        st = [a + b / nf for a, b in zip(st, enc.stage_times())]
        enc.result_size()
    enc.stage_timing(False)
    enc.close()
    # throughput: two encoders on two streams, frames alternating - the offset scan and the compaction of frame n run beside the entropy kernel of
    # frame n + 1, as they do in the GPUJPEG module (one encoder per lane).  Wall clock between two device synchronisations, max over ranks.
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    encs = [api.JpegEncoder(stream=st) for st in streams]
    for e in encs:
        for f in frames:
            e.encode_device(f, W8K, H8K, codec, quality=90)
            e.result_size()
    ctx.barrier()
    n2 = max(48, int(0.35 / per) // 2 * 2)
    t0 = time.perf_counter()
    for i in range(n2):
        encs[i & 1].encode_device(frames[i % nf], W8K, H8K, codec, quality=90)
    torch.cuda.synchronize()
    per2 = ctx.max_over_ranks(time.perf_counter() - t0) / n2
    for e in encs:
        e.result_size()
        e.close()
    single = per
    per = min(per, per2)
    algo = PX * bpp + stream_bytes
    hosts = [host_copy(ctx, frames[i]) for i in range(min(nf, 3))]

    def check(view):  # a stream of the expected size came back through the module
        assert min(sizes) * 0.9 <= view.size <= max(sizes) * 1.1, (view.size, sizes)
    e2e = module_e2e(ctx, "GPUJPEG:q=90", hosts, W8K, H8K, codec, 160 if codec == UYVY else 110, 3, check)
    kname = "ugb::jpeg_fused_kernel<%d,*> + jpeg_scan_kernel + jpeg_compact_kernel" % (0 if codec == UYVY else 1)
    return {"metric": f"7680x4320 frames/sec encode ({'UYVY' if codec == UYVY else 'RGB'}->JPEG q=90)", "value": ctx.world / per, "unit": "frames/s",
            "ms_per_frame": per * 1e3, "single_stream_ms_per_frame": single * 1e3, "two_stream_ms_per_frame": per2 * 1e3,
            "config": {"workload": cfg_note, "frames": nf, "content": "ramps + uniform noise +-6 per channel ('natural'), distinct per frame",
                       "stream_bytes_per_frame": stream_bytes,
                       "pipelining": "value = frames of two encoders alternating on two CUDA streams (as the module's lanes do); single_stream_ms_per_frame = one encoder, "
                                     "its three kernels back to back"},
            "roofline": roofline(ctx, algo, per, kname, f"{name}_bytes_per_frame",
                                 us_blocks=st[0], us_assemble=st[1], us_scan=st[2], us_compact=st[3],
                                 blocks_kernel_achieved=algo / (st[0] * 1e-6) / 1e9 if st[0] > 0 else None,
                                 note="achieved = (input + stream bytes) / whole encode (3 kernels: fused DCT + entropy + segment assembly, offset scan, "
                                      "compaction; us_assemble is non-zero only in the two-kernel form); the kernels are issue- and latency-bound, not HBM-bound"),
            "e2e": {"value": e2e, "unit": "frames/s", "h2d_bytes_per_frame": PX * bpp, "d2h_bytes_per_frame": stream_bytes,
                    "path": "compress_init('GPUJPEG:q=90'), pinned host frame in, stream into a pooled pinned frame, 3 lanes (frames in flight) per device"},
            "gpu_launches_per_frame": 3}


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        reference_arm(args, rank)
        return

    import torch
    import torch.distributed as dist
    from ultragrid_b200 import api, compress, sharding  # raises if libugb200.so is missing: no fallback

    assert torch.cuda.is_available(), "bench.py needs a GPU"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa = api.bind_host_to_device(local_rank)  # before any pinned allocation and before the modules start their threads
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    ctx = Ctx()
    ctx.torch, ctx.api, ctx.compress, ctx.dev, ctx.rank, ctx.local_rank, ctx.world = torch, api, compress, dev, rank, local_rank, world
    ctx.peak, ctx.peak_src = measured_peaks()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(v):
        t = torch.tensor([v], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())
    ctx.barrier, ctx.max_over_ranks = barrier, max_over_ranks
    compress.set_cuda_devices([local_rank])

    B, P, K, Wm = args.frames, args.passes, args.steps, max(args.warmup, 3)
    frame_bytes, out_bytes = PX * 2, PX // 2
    # B distinct noise frames (worst case for DXT: no flat-block shortcut), resident in HBM
    g = torch.Generator(device=dev)
    g.manual_seed(1234 + rank)
    frames = torch.randint(0, 256, (B, frame_bytes), dtype=torch.uint8, device=dev, generator=g)
    outs = torch.empty((B, out_bytes), dtype=torch.uint8, device=dev)
    fr = [frames[f] for f in range(B)]
    ou = [outs[f] for f in range(B)]

    # ---- frame-index assignment: rank 0 owns the queue and scatters int32 indices (the only collective) --------------------------------------
    comm = torch.cuda.Stream(device=dev)
    assign = [torch.zeros(B, dtype=torch.int32, device=dev) for _ in range(2)]
    assign_host = [torch.zeros(B, dtype=torch.int32).pin_memory() for _ in range(2)]
    ready = [torch.cuda.Event() for _ in range(2)]

    def scatter_assignment(step):
        with torch.cuda.stream(comm):
            sharding.scatter_assignment(step, B, assign[step % 2])  # NCCL scatter from rank 0 (a copy when world == 1)
            assign_host[step % 2].copy_(assign[step % 2], non_blocking=True)
            ready[step % 2].record(comm)

    def local_slots(step):
        """what arrived for `step`: global frame indices -> the local batch slots, in queue order (the wait is on an event recorded a whole
        step earlier, so it never blocks the encode)"""
        ready[step % 2].synchronize()
        idx = assign_host[step % 2].numpy()
        base = (step * world + rank) * B
        slots = [int(v) - base for v in idx]
        assert sorted(slots) == list(range(B)), f"rank {rank} step {step}: frame indices {idx[:4]}... are not this rank's share of the queue"
        return slots

    graph, graph_order, enc_stream = None, None, torch.cuda.Stream(device=dev)

    def build_graph(order):
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.stream(enc_stream):
            with torch.cuda.graph(gr, stream=enc_stream, capture_error_mode="thread_local"):
                for f in order:
                    api.uyvy_to_dxt(fr[f], W8K, H8K, dxt_type=1, out=ou[f])
        return gr

    def run_step(step):
        nonlocal graph, graph_order
        scatter_assignment(step + 1)          # next step's assignment travels while this one encodes
        order = local_slots(step)
        if order != graph_order:              # the launch order IS the received assignment
            enc_stream.synchronize()
            graph, graph_order = build_graph(order), order
        with torch.cuda.stream(enc_stream):
            for _ in range(P):
                graph.replay()

    try:
        uuid = str(torch.cuda.get_device_properties(dev).uuid)
    except Exception:
        uuid = None
    clocks = ClockSampler(uuid, local_rank)
    if rank == 0:
        clocks.start()  # NVML initialises while the warm-up runs; only samples inside the timed window are kept
    for f in range(2):  # context / module load outside any capture
        api.uyvy_to_dxt(fr[f], W8K, H8K, dxt_type=1, out=ou[f])
    torch.cuda.synchronize()
    scatter_assignment(0)
    for s in range(Wm):
        run_step(s)
    enc_stream.synchronize()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    clocks.window_begin()
    e0.record(enc_stream)
    for s in range(K):
        run_step(Wm + s)
    e1.record(enc_stream)
    enc_stream.synchronize()
    barrier()
    clocks.window_end()
    ms = e0.elapsed_time(e1)
    clk = clocks.stop() if rank == 0 else None
    ms_max = max_over_ranks(ms)
    fps = world * B * P * K / (ms_max * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_dxt1(outs, args.dump_outputs)

    # ---- end to end through the reference-facing plugin: compress_init("cuda_dxt:DXT1") with pinned HOST frames -------------------------------
    hosts = [host_copy(ctx, frames[i]) for i in range(6)]

    def check_dxt(view):
        assert view.size == out_bytes
    n_e2e = 48 * max(3, min(K, 10))
    e2e_fps = module_e2e(ctx, "cuda_dxt:DXT1", hosts, W8K, H8K, UYVY, n_e2e, 3, check_dxt)

    line = None
    if rank == 0:
        per_launch = ms_max * 1e-3 / (B * P * K)
        line = {
            "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": world, "steps": K,
            "warmup": Wm, "ms_per_step": ms_max / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": {"workload": "7680x4320 UYVY->DXT1 fused encode (ugb200_uyvy_to_dxt1_async), uniform-noise frames",
                       "frames_per_pass_per_gpu": B, "passes_per_step": P, "global_frames_per_step": world * B * P,
                       "l2": f"inputs larger than L2: {B} distinct 66 MB frames per GPU, cycled", "parallelism": f"frame-sharded x{world}",
                       "collective": "NCCL scatter of int32 frame indices, one step ahead on a side stream; encode order built from the received indices",
                       "launch": "one CUDA graph per pass (B kernel nodes)", "numa_node_of_rank0": numa,
                       "other_configs": "see `workloads`: uyvy_jpeg_8k_q90, rgb_jpeg_8k_q90 (config 3), uyvy_dxt5ycocg_8k (config 5), v210_p010_8k (config 4)"},
            "roofline": roofline(ctx, ALGO["uyvy_dxt1"], per_launch, "ugb::dxt_uyvy_kernel<1,2,false>", "dxt_uyvy_kernel_8k_bytes_per_launch"),
            "e2e": {"value": e2e_fps, "unit": "frames/s", "h2d_bytes_per_step": B * P * frame_bytes, "d2h_bytes_per_step": B * P * out_bytes,
                    "frames_timed_per_gpu": n_e2e, "h2d_GBps_per_gpu": e2e_fps / world * frame_bytes / 1e9,
                    "path": "compress_init('cuda_dxt:DXT1'): pinned host UYVY frame (on the GPU's NUMA node) -> compress_frame (H2D, fused kernel, D2H "
                            "into a pooled pinned frame) -> compress_pop; asynchronous module, 3 frames in flight on 3 streams"},
            "gpu_launches": B * P * K,
            "clocks": clk,
        }

    # ---- the other BASELINE workloads, same shape, every N --------------------------------------------------------------------------------------
    if not args.no_extra:
        only = [s for s in args.only.split(",") if s]
        wl = {}

        def guarded(name, fn, *a):  # a failing secondary measurement must not cost the headline line (all ranks take the same path)
            if only and name not in only:
                return
            try:
                wl[name] = fn(*a)
            except Exception as e:  # noqa: BLE001
                wl[name] = {"error": f"{type(e).__name__}: {e}"[:300]}
                try:
                    torch.cuda.synchronize()
                except Exception:  # noqa: BLE001
                    pass
        guarded("uyvy_dxt5ycocg_8k", wl_dxt5, ctx, fr)
        del hosts
        guarded("v210_p010_8k", wl_p010, ctx)
        rgbs = uyvys = None
        try:
            rgbs, uyvys = natural_frames(ctx, 4)
        except Exception as e:  # noqa: BLE001
            wl["natural_frames"] = {"error": str(e)[:200]}
        if uyvys is not None:
            guarded("uyvy_jpeg_8k_q90", wl_jpeg, ctx, "uyvy_jpeg_8k_q90", UYVY, uyvys,
                    "metric, second half: 8K UYVY->JPEG q=90 (4:2:2, one interleaved scan, restart interval 4)")
            guarded("rgb_jpeg_8k_q90", wl_jpeg, ctx, "rgb_jpeg_8k_q90", RGB, rgbs,
                    "BASELINE config 3: 8K RGB->JPEG q=90 (stored as RGB, 4:4:4, three scans, restart interval 8; gpujpeg.cpp:303-305)")
        if rank == 0:
            if world == 1:
                # N = 1 extras first (secondary kernels, decode side, the reference's own GPU kernels): the JPEG decoder's host half must not share
                # the process's CPU quota with the OpenMP team of the CPU baselines that follow
                line["extra"] = {}
                for nm, fn in (("kernels", extra_kernels), ("decode", extra_decode), ("reference_gpu_kernels", reference_gpu_kernels)):
                    try:
                        line["extra"][nm] = fn(ctx)
                    except Exception as e:  # noqa: BLE001
                        line["extra"][nm] = {"error": f"{type(e).__name__}: {e}"[:300]}
                # CPU baselines: rank 0 at N = 1 only, on every CPU the launcher gave us (not just the GPU's NUMA node)
                os.sched_setaffinity(0, LAUNCH_AFFINITY)
                api.bind_host_to_device(-1)
                import util
                cpus = effective_cpus()  # before libgomp loads (see reference_arm)
                orc, ref = util.oracle(), util.ref_cpu()
                orc.orc_set_threads(cpus["used"])
                try:
                    line["cpu_baseline"] = cpu_baseline_block("uyvy_dxt1", orc, ref, cpus, budget_s=6.0)
                except Exception as e:  # noqa: BLE001
                    line["cpu_baseline"] = {"value": None, "unit": "frames/s", "cores": None, "kind": "port", "sample": f"failed: {e}"[:200]}
                cpu_frames = None
                if uyvys is not None:
                    cpu_frames = (uyvys[0].cpu().numpy(), rgbs[0].cpu().numpy())
                for key, nm in (("uyvy_jpeg_8k_q90", "uyvy_jpeg"), ("rgb_jpeg_8k_q90", "rgb_jpeg"), ("uyvy_dxt5ycocg_8k", "uyvy_dxt5"), ("v210_p010_8k", "v210_p010")):
                    if key in wl and "error" not in wl[key]:
                        try:
                            wl[key]["cpu_baseline"] = cpu_baseline_block(nm, orc, ref, cpus, cpu_frames, budget_s=4.0)
                        except Exception as e:  # noqa: BLE001
                            wl[key]["cpu_baseline"] = {"value": None, "sample": f"failed: {e}"[:200]}
                try:
                    line["extra"]["cpu_reference_pixfmt"] = cpu_reference_pixfmt()
                except Exception as e:  # noqa: BLE001
                    line["extra"]["cpu_reference_pixfmt"] = {"error": f"{type(e).__name__}: {e}"[:300]}
            line["workloads"] = wl
            # the headline blocks also list the second half of the metric, so that a reader of only the standard keys sees it
            j = wl.get("uyvy_jpeg_8k_q90", {})
            if "roofline" in j:
                line["roofline"]["uyvy_jpeg_8k_q90"] = {k: j["roofline"][k] for k in ("achieved", "frac", "us_per_launch", "us_blocks", "us_assemble", "us_scan", "us_compact",
                                                                                      "algorithmic_bytes_per_launch", "traffic")}
                line["roofline"]["uyvy_jpeg_8k_q90"]["frames_per_s"] = j["value"]
                line["e2e"]["uyvy_jpeg_8k_q90"] = {"value": j["e2e"]["value"], "unit": "frames/s"}
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


# =====================================================================================================================
# N = 1 extras: secondary kernels, decode side, the reference's own CPU / GPU code beside the product
# =====================================================================================================================
def extra_kernels(ctx):
    """secondary kernels of the path (kernel-only, device-resident, distinct buffers cycled so that L2 does not help)"""
    torch, api, dev = ctx.torch, ctx.api, ctx.dev
    from ultragrid_b200 import Codec, vc_get_linesize
    res = {}

    def rec(name, secs, nbytes, px):
        res[name] = {"us": secs * 1e6, "GBps": nbytes / secs / 1e9, "frac_of_peak": nbytes / secs / 1e9 / ctx.peak, "fps": 1.0 / secs,
                     "bytes_per_px": nbytes / px}

    def rnd(n, count):
        return [torch.randint(0, 256, (n,), dtype=torch.uint8, device=dev) for _ in range(count)]

    # config 2: 3840x2160 UYVY -> DXT1
    w, h = 3840, 2160
    src, out = rnd(w * h * 2, 12), torch.empty(w * h // 2, dtype=torch.uint8, device=dev)
    rec("uyvy_dxt1_4k", graph_timed(ctx, lambda i: api.uyvy_to_dxt(src[i % 12], w, h, out=out), 60, 8), w * h * 2.5, w * h)
    del src
    # reference-ABI RGB -> DXT1 at 8K (the entry point synchronises its stream, like the reference's)
    w, h = W8K, H8K
    src, out = rnd(w * h * 3, 4), torch.empty(w * h // 2, dtype=torch.uint8, device=dev)
    rec("rgb_dxt1_8k_sync_abi", dev_timed(ctx, lambda i: api.compat_to_dxt("cuda_rgb_to_dxt1", src[i % 4], w, h, out=out), 12), w * h * 3.5, w * h)
    import ctypes
    from ultragrid_b200 import _lib
    L = _lib.load()
    rec("rgb_dxt1_8k_async", graph_timed(ctx, lambda i: L.ugb200_rgb_to_dxt1_async(ctypes.c_void_p(src[i % 4].data_ptr()), ctypes.c_void_p(out.data_ptr()), w, h,
                                                                               ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)), 8, 8), w * h * 3.5, w * h)
    del src
    # config 1 on the GPU + 8K line conversions
    for name, inc, outc, ww, hh, n in (("uyvy_rgb_1080p", Codec.UYVY, Codec.RGB, 1920, 1080, 64), ("uyvy_rgb_8k", Codec.UYVY, Codec.RGB, w, h, 4),
                                       ("rgb_uyvy_8k", Codec.RGB, Codec.UYVY, w, h, 4), ("v210_uyvy_8k", Codec.v210, Codec.UYVY, w, h, 4),
                                       ("v210_rgb_8k", Codec.v210, Codec.RGB, w, h, 4), ("uyvy_rgba_8k", Codec.UYVY, Codec.RGBA, w, h, 4)):
        src = rnd(vc_get_linesize(ww, inc) * hh, n)
        dst = torch.empty(vc_get_linesize(ww, outc) * hh, dtype=torch.uint8, device=dev)
        nbytes = (vc_get_linesize(ww, inc) + vc_get_linesize(ww, outc)) * hh
        if ww < 3000:
            secs = graph_timed(ctx, lambda i: api.pixfmt_convert(inc, outc, src[i % n], ww, hh, dst=dst), 64, 8)
        else:
            secs = dev_timed(ctx, lambda i: api.pixfmt_convert(inc, outc, src[i % n], ww, hh, dst=dst), 40)
        rec(name, secs, nbytes, ww * hh)
        del src
    return res


def extra_decode(ctx):
    """decode side (SURVEY 8f rank 1), 8K: kernel-only where the input is device-resident; the JPEG decoder takes a HOST stream
    (parse + upload + kernels), so that number is wall clock per frame"""
    import util
    torch, api, dev = ctx.torch, ctx.api, ctx.dev
    res = {}
    w, h = W8K, H8K
    for t, name in ((1, "dxt1_rgb_8k"), (6, "dxt5ycocg_rgb_8k")):
        nb = w * h // (2 if t == 1 else 1)
        blocks = [torch.randint(0, 256, (nb,), dtype=torch.uint8, device=dev) for _ in range(4)]
        out = torch.empty(w * h * 3, dtype=torch.uint8, device=dev)
        secs = dev_timed(ctx, lambda i: api.dxt_to_rgb(blocks[i % 4], w, h, t, out=out), 12)
        res[name] = {"us": secs * 1e6, "fps": 1 / secs, "GBps": (nb + w * h * 3) / secs / 1e9, "frac_of_peak": (nb + w * h * 3) / secs / 1e9 / ctx.peak}
        del blocks
    orc = util.oracle()
    uyvy, rgb = _natural_uyvy_cpu(orc)
    # UYVY: one interleaved scan (what UltraGrid sends for UYVY input); RGB: one scan per component, as GPUJPEG stores RGB (config 3 on the receiving side)
    for name, codec, frame in (("jpeg_decode_natural_8k", UYVY, uyvy), ("jpeg_decode_rgb_natural_8k", RGB, rgb)):
        enc = api.JpegEncoder()
        enc.encode_device(torch.from_numpy(frame).cuda(), w, h, codec, quality=90)
        stream = enc.result()
        enc.close()
        dec = api.JpegDecoder()
        out = dec.decode(stream, codec, device=True)
        for _ in range(3):  # both host slots have their pinned staging, the scratch vectors their capacity
            dec.decode(stream, codec, device=True, out=out, sync=False)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        n = 16
        for _ in range(n):
            dec.decode(stream, codec, device=True, out=out, sync=False)
        torch.cuda.synchronize()
        res[name] = {"ms_wall_per_frame": (time.perf_counter() - t0) / n * 1e3, "stream_bytes": len(stream),
                     "output": ("UYVY" if codec == UYVY else "RGB") + " on the device; host stream in (marker scan on the device, upload on a copy stream)"}
        dec.close()
        del out
    return res


def reference_gpu_kernels(ctx):
    """SURVEY 8d: for the DXT configs the reference beside the product is its own CUDA path — the UNMODIFIED cuda_dxt.cu built for
    sm_100a (oracle/_ref/libcuda_dxt_ref.so), i.e. cuda_yuv422_to_yuv444 + cuda_yuv_to_dxt{1,6} as src/video_compress/cuda_dxt.cpp
    :229,257 runs them (each call synchronises its stream, cuda_dxt.cu:759).  Baseline only; never part of `value`."""
    import ctypes
    import util
    torch, dev = ctx.torch, ctx.dev
    ref = util.ref_gpu()
    if ref is None:
        return {"unavailable": "oracle/_ref/libcuda_dxt_ref.so not present"}
    w, h = W8K, H8K
    srcs = [torch.randint(0, 256, (w * h * 2,), dtype=torch.uint8, device=dev) for _ in range(3)]
    mid = torch.empty(w * h * 3, dtype=torch.uint8, device=dev)
    out = torch.empty(w * h, dtype=torch.uint8, device=dev)
    res = {}
    for name, fn in (("uyvy_dxt1_8k", ref.cuda_yuv_to_dxt1), ("uyvy_dxt5ycocg_8k", ref.cuda_yuv_to_dxt6)):
        def step(i):
            ref.cuda_yuv422_to_yuv444(ctypes.c_void_p(srcs[i % 3].data_ptr()), ctypes.c_void_p(mid.data_ptr()), w * h, None)
            fn(ctypes.c_void_p(mid.data_ptr()), ctypes.c_void_p(out.data_ptr()), w, h, None)
        for i in range(2):
            step(i)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        n = 6
        for i in range(n):
            step(i)
        torch.cuda.synchronize()
        secs = (time.perf_counter() - t0) / n
        res[name] = {"us": secs * 1e6, "fps": 1 / secs}
    return res


def cpu_reference_pixfmt():
    """the reference's own CPU pixfmt_conv path (unmodified objects in oracle/_ref) on this host: UYVY->RGB (BASELINE config 1 at 1080p, and
    8K), 1 thread and all cores through parallel_pix_conv (src/utils/parallel_conv.c:64-85)"""
    import numpy as np
    import util
    ref = util.ref_cpu()
    if ref is None:
        return {"unavailable": "oracle/_ref/libugref.so not present"}
    out = {"cpus": effective_cpus(), "flags": "-O3 -msse4.1 (tools/Makefile)"}
    for tag, w, h in (("1080p", 1920, 1080), ("8k", W8K, H8K)):
        src = util.rng_bytes(w * h * 2, 9)
        dst = np.zeros(w * h * 3, dtype=np.uint8)
        for label, fn in (("1_thread", lambda: ref.ref_convert(UYVY, RGB, dst.ctypes.data, w * 3, src.ctypes.data, w * 2, w * 3, h, 0, 8, 16)),
                          ("all_cores", lambda: ref.ref_convert_parallel(UYVY, RGB, dst.ctypes.data, w * 3, src.ctypes.data, w * 2, h, 0))):
            best, med, n = time_cpu(fn, budget_s=2.0)
            out[f"uyvy_rgb_{tag}_{label}_ms"] = {"best": best * 1e3, "median": med * 1e3, "runs": n}
    return out


if __name__ == "__main__":
    main()
