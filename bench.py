#!/usr/bin/env python3
"""bench.py — throughput of the H.264 reconstruction path on B200 (contract: see the task statement).

Workloads (synthetic Annex-B streams written on the spot by tools/gen264, fixed seeds):
  --config 1080p (default)  BASELINE.json configs[1]: 1080p High CABAC I/P/B ~30 Mbit/s, 32 streams x 60 frames per GPU
  --config 2160p            configs[2]: 3840x2160, 8x8 transform + custom quantisation matrices, 8 streams x 16 frames per GPU
  --config 4320p            configs[4]: 7680x4320 level 6.2, B slices with explicit weighted bi-prediction, every edge
                            filtered; ONE stream of closed GOPs (I P B P), cut at its IDR pictures on rank 0 and sharded
                            BY GOP over the ranks (4 GOPs per GPU), each GOP decoded by its own decoder instance
One "step" = one pass over the batch of one GPU.

  value   kernel-only replay: the batch's per-macroblock records are resident in HBM, every picture's kernels are re-run in
          decode order on one CUDA stream per decoder, timed with CUDA events.  A stream's pictures of one step are one
          CUDA graph (same kernels, same order; one graph launch per stream and step) so that the host's launch rate
          does not bound a device number; E264B_REPLAY_GRAPH=0 issues the launches one by one from several host threads.
          Each launch also stamps its first/last block (%globaltimer): the roofline object is computed from THIS pass.
  e2e     the same batch decoded through the edge264 C API (edge264_decode_NAL / get_frame) from HOST buffers: CPU
          parsing, H2D of the records, kernels, D2H of every frame and a host read of every output frame are inside the
          timed region.  A pool of application threads (one per usable CPU, at most one per stream) takes the streams one
          after the other; with CPUs to spare each decoder also parses ahead on worker threads (edge264_alloc n_threads).
  --impl reference   the reference decoder compiled from its own sources (oracle/_ref), one single-threaded decoder per
          stream on all usable host cores, same streams, same application loop.
  --dump-outputs DIR  after the timed steps, what the decode loop handed to the application in its last timed step (the
          kernel-only replay re-runs the kernels of exactly these pictures): a fixed, seeded choice of output frames
          (DUMP_FRAMES at most) and of sample positions in them, so that two builds can be compared output for output.
            DIR/frames.npy      float32 [frames, positions]: 8-bit samples of the cropped Y, Cb and Cr planes laid end to end
            DIR/frame_info.npy  float64 [frames, 7]: unit, index in output order, FrameId, width_Y, height_Y, width_C, height_C
"""
import argparse, ctypes, hashlib, json, os, subprocess, sys, tempfile, threading, time

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
ROOT = os.path.dirname(os.path.abspath(__file__))

CONFIGS = {
    "1080p": {"metric": "1080p_high_cabac_ipb_decode_fps", "w": 120, "h": 68, "frames": 60, "streams": 32, "seed0": 2000,
              "workload": "1080p High CABAC IPB ~30 Mbit/s (BASELINE configs[1])", "unit_of_sharding": "stream",
              "gen": "--gop IPB --idr 30 --refs 2 --t8x8 50 --deblock 0 --density 52 --qp 28 --wp 0"},
    "2160p": {"metric": "2160p_high_8x8_scaling_decode_fps", "w": 240, "h": 135, "frames": 16, "streams": 8, "seed0": 3000,
              "workload": "3840x2160 High, 8x8 transform + custom quantisation matrices (BASELINE configs[2])", "unit_of_sharding": "stream",
              "gen": "--gop IPB --idr 16 --refs 2 --t8x8 70 --scaling 3 --deblock 0 --density 40 --qp 30 --wp 0"},
    "4320p": {"metric": "4320p_wp_bipred_decode_fps", "w": 480, "h": 270, "frames": 4, "streams": 4, "seed0": 4000,
              "workload": "7680x4320 level 6.2, B slices with explicit weighted bi-prediction, all edges filtered, closed GOPs of 4 (BASELINE configs[4])", "unit_of_sharding": "closed GOP of one stream",
              "gen": "--gop IPB --idr 4 --refs 2 --wp 1 --deblock 0 --density 60 --skip-pct 0"},
}


def generate_streams(cfg, seeds, frames, workdir):
    os.makedirs(workdir, exist_ok=True)
    gen = os.path.join(ROOT, "tools", "gen264")
    if not os.path.exists(gen):
        raise SystemExit("tools/gen264 missing: run `python -c 'import __graft_entry__ as g; g.build()'` first")
    # a cached stream is named after the generator binary and its arguments and appears only once complete, so the inputs
    # are what this build's generator writes for these arguments, never a file of another build or of an interrupted run
    key = hashlib.sha1(open(gen, "rb").read() + cfg["gen"].encode()).hexdigest()[:12]
    procs, paths = [], []
    def finish(procs):
        for q, part, p in procs:
            if q.wait() != 0:
                raise SystemExit(f"bench.py: tools/gen264 failed on {p}")
            os.replace(part, p)
    for s in seeds:
        p = os.path.join(workdir, f"{cfg['w']}x{cfg['h']}_{s}_{frames}_{key}.264")
        paths.append(p)
        if not os.path.exists(p):
            part = f"{p}.{os.getpid()}.part"
            procs.append((subprocess.Popen([gen, "-o", part, "-W", str(cfg["w"]), "-H", str(cfg["h"]), "-n", str(frames), "-s", str(s)] + cfg["gen"].split(), stderr=subprocess.DEVNULL), part, p))
        if len(procs) >= 16:
            finish(procs); procs = []
    finish(procs)
    return [open(p, "rb").read() for p in paths]


def batch_for(cfg, n_units, workdir, frames):
    """The input of `n_units` sharding units.  Streams: one generated stream each.  GOPs: ONE long stream (the closed GOPs
    of independent seeds concatenated: every GOP starts with SPS, PPS and an IDR picture), cut again at its IDR pictures
    the way a real input would be."""
    bufs = generate_streams(cfg, [cfg["seed0"] + i for i in range(n_units)], frames, workdir)
    if cfg["unit_of_sharding"] == "stream":
        return bufs
    from edge264_b200.shard import split_closed_gops
    gops = split_closed_gops(b"".join(bufs))
    assert len(gops) == n_units, (len(gops), n_units)
    return gops


class BenchLib:
    def __init__(self, path):
        self.lib = ctypes.CDLL(path)
        self.lib.e264bench_run.restype = ctypes.c_double
        self.lib.e264bench_run.argtypes = [ctypes.POINTER(ctypes.c_char_p), ctypes.POINTER(ctypes.c_size_t), ctypes.c_int, ctypes.c_int,
                                            ctypes.c_int, ctypes.POINTER(ctypes.c_long), ctypes.POINTER(ctypes.c_uint64), ctypes.POINTER(ctypes.c_void_p)]
        self.lib.e264bench_free.argtypes = [ctypes.POINTER(ctypes.c_void_p), ctypes.c_int]

    def run(self, bufs, threads, keep=False):
        n = len(bufs)
        arr = (ctypes.c_char_p * n)(*bufs)
        sizes = (ctypes.c_size_t * n)(*[len(b) for b in bufs])
        frames = (ctypes.c_long * n)(); sums = (ctypes.c_uint64 * n)(); decs = (ctypes.c_void_p * n)()
        secs = self.lib.e264bench_run(arr, sizes, n, threads, 1 if keep else 0, frames, sums, decs)
        return secs, list(frames), list(sums), decs

    def free(self, decs): self.lib.e264bench_free(decs, len(decs))


DUMP_FRAMES, DUMP_FLOATS, DUMP_SEED = 32, 15 << 20, 264      # --dump-outputs: at most 60 MB of float32 samples


def dump_selection(frames):
    """The output frames --dump-outputs keeps, given the frame count of every unit: a seeded choice of at most DUMP_FRAMES
    of them, as (unit, index in output order)."""
    import numpy as np
    total = sum(frames)
    flat = np.sort(np.random.default_rng(DUMP_SEED).choice(total, min(DUMP_FRAMES, total), replace=False))
    starts = np.cumsum([0] + list(frames[:-1]))
    unit = np.searchsorted(starts, flat, side="right") - 1
    return unit.astype(np.int32), (flat - starts[unit]).astype(np.int64)


class Capture:
    """--dump-outputs: the selected output frames are copied by the decode loop itself (e264bench_capture) while the
    capture is on; write() stores a seeded choice of sample positions of them."""
    def __init__(self, bench, frames, cfg):
        import numpy as np
        # bound here, not in BenchLib: a driver library built before the capture existed still serves every other use
        if not hasattr(bench.lib, "e264bench_capture"):
            raise SystemExit(f"bench.py --dump-outputs: {bench.lib._name} has no e264bench_capture; rebuild it from tools/e264_bench.c")
        bench.lib.e264bench_capture.argtypes = [ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p]
        self.bench, self.unit, self.index = bench, *dump_selection(frames)
        n, cap = len(self.unit), cfg["w"] * cfg["h"] * 384
        self.buf = np.zeros((n, cap), np.uint8); self.info = np.full((n, 5), -1, np.int32)
        self.dst = (ctypes.c_void_p * n)(*[self.buf[k].ctypes.data for k in range(n)])
        bench.lib.e264bench_capture(n, self.unit.ctypes.data, self.index.ctypes.data, self.dst, cap, self.info.ctypes.data)

    def stop(self):
        self.bench.lib.e264bench_capture(0, None, None, None, 0, None)

    def write(self, out):
        import numpy as np
        assert (self.info[:, 0] >= 0).all(), "a frame chosen for --dump-outputs was not delivered"
        size = int(min(wy * hy + 2 * wc * hc for _, wy, hy, wc, hc in self.info))
        pos = np.sort(np.random.default_rng(DUMP_SEED + 1).choice(size, min(size, DUMP_FLOATS // len(self.unit)), replace=False))
        os.makedirs(out, exist_ok=True)
        np.save(os.path.join(out, "frames.npy"), self.buf[:, pos].astype(np.float32))
        np.save(os.path.join(out, "frame_info.npy"), np.column_stack([self.unit, self.index, self.info]).astype(np.float64))


class ReplayStats(ctypes.Structure):
    _fields_ = [("ms_total", ctypes.c_float), ("threads", ctypes.c_int), ("launches", ctypes.c_uint64),
                ("kernel_ms", ctypes.c_double * 5), ("kernel_launches", ctypes.c_uint64 * 5), ("inflight", ctypes.c_int), ("reserved", ctypes.c_int)]


KERNELS = ["(unused)", "e264_inter4_kernel", "e264_intra_kernel / e264_intra_rows_kernel", "e264_deblock_kernel", "(unused)"]


class ClockSampler(threading.Thread):
    """SM clock and clock-event (throttle) reasons during the timed regions (B200_PROFILING.md recipe).  NVML through
    nvidia_ml_py when it is importable (a query costs microseconds, so the short device-timed replay gets tens of samples and
    the CPU-bound e2e phase loses nothing to the sampler); otherwise one nvidia-smi process per second."""
    def __init__(self, gpu):
        super().__init__(daemon=True); self.gpu = gpu; self.rows = []; self.stop = False; self.period = 0.5; self.nvml = None; self.h = None; self.wake = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit(); self.h = pynvml.nvmlDeviceGetHandleByIndex(gpu); self.nvml = pynvml
        except Exception:
            self.nvml = None
    def sample(self):
        if self.nvml is not None:
            n = self.nvml
            sm = n.nvmlDeviceGetClockInfo(self.h, n.NVML_CLOCK_SM); mx = n.nvmlDeviceGetMaxClockInfo(self.h, n.NVML_CLOCK_SM)
            try: r = n.nvmlDeviceGetCurrentClocksEventReasons(self.h)
            except Exception: r = n.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
            act = lambda bit: "Active" if r & bit else "Not Active"
            return [str(sm), str(mx), act(0x8), act(0x40), act(0x20), act(0x4)]      # hw_slowdown, hw_thermal, sw_thermal, sw_power_cap
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        o = subprocess.run(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={q}", "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout.strip()
        return [x.strip() for x in o.split(",")] if o else None
    def run(self):
        while not self.stop:
            try:
                r = self.sample()
                if r: self.rows.append(r + [self.phase])
            except Exception:
                pass
            self.wake.wait(self.period if self.nvml is not None else max(self.period, 1.0)); self.wake.clear()
    phase = "e2e"
    def set_phase(self, phase, period):
        self.phase = phase; self.period = period; self.wake.set()
    def summary(self):
        if not self.rows: return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}
        rows = [r for r in self.rows if r[-1] == "replay"] or self.rows      # the device-timed region when it was sampled
        sm = sorted(int(r[0]) for r in rows if r[0].isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[2 + i].lower().startswith("active") for r in self.rows if len(r) > 3 + i)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": int(self.rows[0][1]) if self.rows[0][1].isdigit() else None, "reasons": reasons,
                "samples": len(self.rows), "samples_in_replay": sum(1 for r in self.rows if r[-1] == "replay"), "source": "nvml" if self.nvml is not None else "nvidia-smi"}


def usable_cpus():
    """CPUs this container may actually use: min(affinity, cgroup quota) — the 1-GPU boxes grant 16 of 128."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max": n = min(n, max(1, int(int(q) / int(per) + 0.5)))
    except Exception:
        pass
    return n


def peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"], "measured"
    except Exception:
        return 6650.0, "fallback"


def ncu_traffic(config, group):
    """DRAM bytes per picture ncu saw for this kernel group on the bench streams (profiles/r2_ncu_traffic.json); None if absent."""
    try:
        return float(json.load(open(os.path.join(ROOT, "profiles", "r2_ncu_traffic.json")))[config][group]["dram_bytes_per_picture"])
    except Exception:
        return None


def config_dict(cfg, args, world):
    """Identical for both arms: the driver compares it."""
    return {"workload": f"{cfg['workload']}, {cfg['w'] * 16}x{cfg['h'] * 16}, {args.frames} frames per {cfg['unit_of_sharding']}, {args.streams} per GPU",
            "units_per_gpu": args.streams, "frames_per_unit": args.frames, "unit": cfg["unit_of_sharding"], "n_gpus": world,
            "l2": "working set per step (records + coefficients + frames of all streams) > 126 MB L2",
            "parallelism": f"{cfg['unit_of_sharding']}s sharded over {world} GPU(s), NCCL broadcast of the input only"}


def reference_arm(args, cfg, rank, world, emit):
    """CPU reference decoder on all usable host cores (rank 0 only), same batch as the GPU arm at this N."""
    if rank != 0:
        return
    lib = os.path.join(ROOT, "oracle", "_ref", "libe264bench_ref.so")
    if not os.path.exists(lib):
        emit({"impl": "reference", "unavailable": "oracle/_ref not built (run __graft_entry__.build() where /root/reference exists)"}); return
    ref = BenchLib(lib)
    n_units = args.streams * world
    bufs = batch_for(cfg, n_units, args.workdir, args.frames)
    threads = max(1, min(usable_cpus(), n_units))   # one single-threaded decoder per usable CPU (cgroup quota respected)
    fr = None
    for _ in range(args.warmup): _, fr, _, _ = ref.run(bufs, threads)
    t = 0.0; frames = 0; cap = None
    for step in range(args.steps):
        if args.dump_outputs and step == args.steps - 1:
            cap = Capture(ref, fr or ref.run(bufs, threads)[1], cfg)      # the choice needs every unit's frame count
        s, fr, _, _ = ref.run(bufs, threads)
        t += s; frames += sum(fr)
    if cap is not None:
        cap.stop(); cap.write(args.dump_outputs)
    fps = frames / t
    mbpf = cfg["w"] * cfg["h"]
    line = {"metric": cfg["metric"], "value": fps, "unit": "frames/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1000 * t / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "impl": "reference", "macroblocks_per_s": fps * mbpf, "config": config_dict(cfg, args, world),
            "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": threads, "kind": "reference",
                             "sample": f"{n_units} {cfg['unit_of_sharding']}s x {args.frames} frames per step, n_threads=0 decoders, {threads} worker threads of {usable_cpus()} usable CPUs"},
            "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


def main():
    # stdout carries exactly ONE JSON line: libraries that print there (NCCL's version banner) are diverted to stderr
    real_stdout = os.dup(1); os.dup2(2, 1)
    def emit(obj):
        os.write(real_stdout, (json.dumps(obj) + "\n").encode())
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1); ap.add_argument("--steps", type=int, default=5); ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200"); ap.add_argument("--config", default="1080p", choices=sorted(CONFIGS))
    ap.add_argument("--streams", type=int, default=0, help="sharding units (streams or GOPs) per GPU; 0 = the config's default")
    ap.add_argument("--frames", type=int, default=0, help="frames per unit; 0 = the config's default")
    ap.add_argument("--dec-threads", type=int, default=-1, help="edge264_alloc n_threads of every decoder; -1 = from the CPUs available per stream")
    ap.add_argument("--workdir", default=os.environ.get("E264_BENCH_DIR", os.path.join(tempfile.gettempdir(), f"e264_bench_{os.getuid()}")))
    ap.add_argument("--dump-outputs", metavar="DIR", help="write a seeded sample of the last timed step's output frames to DIR (see the module docstring)")
    args = ap.parse_args()
    cfg = CONFIGS[args.config]
    if args.streams <= 0: args.streams = cfg["streams"]
    if args.frames <= 0: args.frames = cfg["frames"]
    rank = int(os.environ.get("RANK", "0")); local = int(os.environ.get("LOCAL_RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        reference_arm(args, cfg, rank, world, emit); return

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the reconstruction path has no CPU fallback")
    torch.cuda.set_device(local)
    os.environ["E264B_DEVICE"] = str(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    S, F = args.streams, args.frames
    mbpf = cfg["w"] * cfg["h"]
    # rank 0 owns the input (for the GOP config: cuts the one stream at its IDR pictures) and broadcasts it over NCCL
    bufs_all = batch_for(cfg, S * world, args.workdir, F) if rank == 0 else None
    from edge264_b200.shard import broadcast_streams, max_over_ranks
    bufs = broadcast_streams(bufs_all, S, world, rank, dist, "cuda")

    # host threads: one application thread per unit (it sleeps while its decoder waits); with CPUs to spare every decoder
    # also parses ahead on worker threads
    cpus = max(1, usable_cpus() // world)
    dec_threads = args.dec_threads if args.dec_threads >= 0 else max(0, min(4, cpus // S))
    os.environ["E264_BENCH_DEC_THREADS"] = str(dec_threads)
    # application threads: a pool that takes the units one after the other, like the reference arm's; no more threads than
    # CPUs (measured on the 16-CPU box, profiles/r2_e2e_threads.txt: 32 units on 16 threads 1292 frames/s, on 32 threads 1220 —
    # the waits for the GPU are short, surplus threads only cost context switches and cache)
    app_threads = max(1, min(S, cpus))

    lib = BenchLib(os.path.join(ROOT, "tools", "libe264bench.so"))
    core = ctypes.CDLL(os.path.join(ROOT, "edge264_b200", "libedge264_b200.so"))
    core.e264b_of_decoder.restype = ctypes.c_void_p; core.e264b_of_decoder.argtypes = [ctypes.c_void_p]
    core.e264b_replay.argtypes = [ctypes.POINTER(ctypes.c_void_p), ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.POINTER(ReplayStats)]
    core.e264b_kept_algorithmic_bytes.restype = ctypes.c_double
    core.e264b_kept_algorithmic_bytes.argtypes = [ctypes.c_void_p, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_uint64)]
    core.e264b_stats.argtypes = [ctypes.c_void_p, ctypes.POINTER(ctypes.c_uint64), ctypes.POINTER(ctypes.c_uint64), ctypes.POINTER(ctypes.c_uint64)]
    core.e264b_error_flag.argtypes = [ctypes.c_void_p]

    def barrier():
        if dist is not None: dist.barrier()
        torch.cuda.synchronize()
    def maxreduce(x): return max_over_ranks(x, dist, "cuda")

    # ---- e2e: decode through the C API from host buffers ----
    os.environ["E264B_KEEP"] = "0"
    # warm-up: the first pass keeps its decoders alive until the end of the pass, so that one device context per unit exists
    # (they are pooled and reused afterwards: no allocation inside the timed region) and the bytes each decoder copied can
    # be read; the passes are identical, so these are the bytes of every timed step as well
    h2d = d2h = 0
    for k in range(max(args.warmup, 1)):
        _, frames, sums, d = lib.run(bufs, app_threads, keep=(k == 0))
        if k == 0:
            for i in range(S):
                a, b, c = ctypes.c_uint64(), ctypes.c_uint64(), ctypes.c_uint64()
                core.e264b_stats(core.e264b_of_decoder(d[i]), ctypes.byref(a), ctypes.byref(b), ctypes.byref(c)); h2d += b.value; d2h += c.value
        lib.free(d)
    frames_per_step = sum(frames)
    sampler = ClockSampler(local); sampler.start()
    barrier()
    e2e_secs = 0.0; cap = None
    for step in range(args.steps):
        if args.dump_outputs and rank == 0 and step == args.steps - 1:
            cap = Capture(lib, frames, cfg)
        s, fr, sm, d = lib.run(bufs, app_threads)      # every decoder is freed as soon as its stream ends, like an application would
        lib.free(d)
        e2e_secs += s
        assert sm == sums, "e2e output differs between runs"
    if cap is not None:
        cap.stop()
    barrier()
    e2e_secs = maxreduce(e2e_secs)
    e2e_fps = world * frames_per_step * args.steps / e2e_secs

    # the same batch once more with E264B_KEEP=1: the decoders stay alive and retain their device-side records
    os.environ["E264B_KEEP"] = "1"
    _, frames, sums_k, decs = lib.run(bufs, app_threads, keep=True)
    assert sums_k == sums
    os.environ["E264B_KEEP"] = "0"
    devs = (ctypes.c_void_p * S)(*[core.e264b_of_decoder(decs[i]) for i in range(S)])

    # ---- kernel-only replay (records resident in HBM): one CUDA graph per stream and step (plain launches: 2 host threads,
    # more of them contend for the driver and issue fewer launches per second in total) ----
    launch_threads = max(1, min(S, cpus, 2))
    st = ReplayStats()
    for _ in range(args.warmup):
        core.e264b_replay(devs, S, 1, launch_threads, ctypes.byref(st))
    barrier()
    sampler.set_phase("replay", 0.005)
    rc = core.e264b_replay(devs, S, args.steps, launch_threads, ctypes.byref(st))
    barrier()
    if rc != 0 or any(core.e264b_error_flag(devs[i]) for i in range(S)):
        raise SystemExit("bench.py: replay failed (CUDA error or dependency timeout)")
    step_ms = maxreduce(st.ms_total) / args.steps
    sampler.stop = True; sampler.wake.set(); sampler.join(timeout=2)
    fps = world * frames_per_step / (step_ms / 1000)

    # ---- roofline from the timed pass: per-launch device spans, algorithmic bytes of SURVEY.md section 8(d) ----
    rb = db = 0.0
    for i in range(S):
        r, d_ = ctypes.c_double(), ctypes.c_double(); n = ctypes.c_uint64()
        core.e264b_kept_algorithmic_bytes(devs[i], ctypes.byref(r), ctypes.byref(d_), ctypes.byref(n)); rb += r.value; db += d_.value
    rb *= args.steps; db *= args.steps                      # bytes of the whole timed region on this GPU
    kms = [st.kernel_ms[k] for k in range(5)]; kn = [int(st.kernel_launches[k]) for k in range(5)]
    groups = {"reconstruction": {"kinds": [1, 2], "bytes": rb}, "deblocking": {"kinds": [3], "bytes": db}}
    for g in groups.values():
        g["ms"] = sum(kms[k] for k in g["kinds"]); g["launches"] = max([kn[k] for k in g["kinds"]] + [1])
    dom = max(groups, key=lambda g: groups[g]["ms"])
    G = groups[dom]
    top = max(G["kinds"], key=lambda k: kms[k])
    peak, how = peaks()
    achieved = G["bytes"] / (G["ms"] / 1000) / 1e9 if G["ms"] > 0 else 0.0
    pictures = S * F * args.steps
    traffic_pp = ncu_traffic(args.config, dom)
    roof = {"bound": "hbm", "kernel": KERNELS[top] + f" (dominant by device time; its group: the {dom} launches of a picture = " + " + ".join(KERNELS[k] for k in G["kinds"]) + ")",
            "achieved": achieved, "peak": peak, "peak_source": how + " (MEASURED_PEAKS.json hbm_gbs)", "unit": "GB/s", "frac": achieved / peak,
            "algorithmic_bytes_per_launch": G["bytes"] / pictures, "avg_launch_ms": G["ms"] / pictures,
            "traffic": traffic_pp,
            "traffic_note": "DRAM read+write bytes per picture of this kernel group from an ncu capture of the same streams (profiles/r2_ncu_traffic.json); algorithmic_bytes_per_launch is the figure `achieved` uses",
            "how": "achieved = algorithmic bytes of the group's launches / sum of their device spans (first block start to last block end, %globaltimer) measured inside the timed replay; launches of different streams overlap, so this is the per-launch (serialised) rate",
            "concurrent": {"achieved": (rb + db) / (st.ms_total / 1000) / 1e9, "frac": (rb + db) / (st.ms_total / 1000) / 1e9 / peak, "note": "all algorithmic bytes of the step / elapsed time of the step, every stream in flight"},
            "per_kernel": {KERNELS[k]: {"launches": kn[k], "sum_ms": kms[k], "avg_us": 1000 * kms[k] / kn[k] if kn[k] else None} for k in (1, 2, 3)},
            "per_group": {g: {"sum_ms": v["ms"], "algorithmic_gb": v["bytes"] / 1e9, "achieved_gbs": v["bytes"] / (v["ms"] / 1000) / 1e9 if v["ms"] > 0 else None} for g, v in groups.items()}}

    line = {"metric": cfg["metric"], "value": fps, "unit": "frames/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": step_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "macroblocks_per_s": fps * mbpf, "config": config_dict(cfg, args, world),
            "clocks": sampler.summary(), "gpu_launches": int(st.launches), "replay": f"cuda-graph per stream and step, {int(st.inflight)} streams in flight" if st.threads == 0 else f"{int(st.threads)} host launch threads",
            "e2e": {"value": e2e_fps, "unit": "frames/s", "macroblocks_per_s": e2e_fps * mbpf, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "app_threads": app_threads, "decoder_n_threads": dec_threads, "usable_cpus": usable_cpus(), "cpus_per_rank": cpus, "bytes_per_unit": len(bufs[0]),
                    "saturated": "host CPUs (bitstream parsing)" if app_threads * max(1, dec_threads + 1) >= cpus else "streams in flight",
                    "note": "edge264_decode_NAL/get_frame from host buffers; bound by the host's CPUs (bitstream parsing) as soon as application threads x (1 + parse-ahead workers) reach the usable CPUs — on one host that is already the case at N = 1, so e2e follows the CPUs, not the number of GPUs; get_frame polls and only waits after ENOBUFS / at the end of a stream"},
            "roofline": roof}
    lib.free(decs)
    if cap is not None:
        cap.write(args.dump_outputs)

    if rank == 0 and world == 1:
        refp = os.path.join(ROOT, "oracle", "_ref", "libe264bench_ref.so")
        if os.path.exists(refp):
            ref = BenchLib(refp)
            threads = max(1, min(usable_cpus(), S))
            # bounded sample: as many units as threads (1080p: ~1 s of work per unit), at most the batch
            rb_ = bufs[:max(1, min(S, threads))]
            s, fr, rs, _ = ref.run(rb_, threads)
            line["cpu_baseline"] = {"value": sum(fr) / s, "unit": "frames/s", "cores": min(threads, len(rb_)), "kind": "reference",
                                    "sample": f"{len(rb_)} {cfg['unit_of_sharding']}s x {F} frames, {min(threads, len(rb_))} single-threaded reference decoders at a time, host of this box ({os.cpu_count()} logical CPUs, {usable_cpus()} usable under the cgroup quota)",
                                    "bit_exact_with_gpu": all(rs[i] == sums[i] for i in range(len(rb_)))}
        else:
            line["cpu_baseline"] = {"value": None, "unit": "frames/s", "cores": 0, "kind": "reference", "sample": "oracle/_ref missing"}
    if rank == 0:
        emit(line)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
