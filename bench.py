#!/usr/bin/env python
"""bench.py — the render hot path on BASELINE.json's headline workload.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A *step* renders one frame of each headline scene — rgbbox 1000x1000 and irreg 1000x1000 at 64 samples
per pixel (BASELINE.json configs[1] and configs[2], the configs its metric "Mrays/s rgbbox+irreg
1000^2" is quoted on) — through the C ABI of libray_b200.so.  A *ray* is one ray segment = one
`objs_hit` call (SURVEY.md §8d); the per-frame segment counts come from the library's counting kernel
and equal the oracle's (tests/test_gpu_parity.py::test_work_counters_equal_reference_traversal).

Prints ONE JSON line (rank 0).
`value` = segments of all frames of K steps / device time (scene resident in HBM, CUDA events on the launch stream, max over
ranks).  Default protocol: the K steps are submitted back to back with pipelined submission (ray_b200_context_set_pipeline:
frames alternate between two lanes across steps, so a frame's last 50-bounce paths are covered by the next frame's start), ONE
event pair around all K steps, the per-step L2 flush inside it; `strict_steps` repeats the K steps in the round-1 protocol
(every step one joined batch between its own event pair) for comparison, `--strict-steps` makes that the headline.
`e2e` = the same through host buffers, wall clock with barrier + synchronize on both sides: per step H2D of every scene's packed
sphere records from pinned memory + LBVH build on the device (every rank), the step's frames as one batch, and every frame's D2H
into pinned host memory (rank 0) through the peer-frame ring (raytracers_b200.distributed.PeerFrameRenderer; at N > 1 the other
ranks' kernels write their pixels straight into rank 0's frame over NVLink) - the delivered host frames are compared with the
oracle in `parity`.  `--gather nccl` switches N > 1 to tile buffers + one ncclGather + de-tiling per frame.
`roofline` = the render kernel's algorithmic bytes (32 B x box tests + 16 B x sphere tests + 4 B x pixels, reference traversal
counts) / its measured duration vs the measured HBM peak - an accounting figure, the scene is shared-memory resident;
`roofline_issue` = useful thread-instructions of the reference traversal / the chip's issue capacity - the bound that applies;
`parity` / `extra.*.parity` = differing pixels between the GPU frames and the oracle's row samples of the SAME frames (timed
workload and the other BASELINE configs), plus - at every N - whether the SHA-256 of the full frames the end-to-end leg
delivered to host memory equals the oracle's known answers (tests/golden/oracle_frame_hashes.json); `cpu_baseline` = the CPU oracle (a bit-exact port of the reference's Futhark program;
the Futhark compiler is not available here) on a bounded sample of the same workload.

--impl reference times that same CPU port on all host cores (no GPU work), one bounded sample per step.
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# the peer-frame path waits on flags with 1-thread kernels; give every stream its own hardware queue (must be set before CUDA starts)
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

SCENES = ("rgbbox", "irreg")
H = W = 1000
SPP = 64
ROW_STEP = 8  # CPU legs render rows j % ROW_STEP == 0 of every frame (a 1/8 sample of the step)
METRIC = "Mrays/s (ray segments/s) rgbbox+irreg 1000x1000"
WORKLOAD = "rgbbox 1000x1000 64spp + irreg 1000x1000 64spp per step (BASELINE.json configs[1]+configs[2])"


def dram_traffic_per_launch():
    """dram__bytes_read.sum + dram__bytes_write.sum per render launch from the committed ncu capture."""
    try:
        with open(os.path.join(ROOT, "profiles", "dram_traffic.json")) as f:
            d = json.load(f)
        return {k: int(d[k]) for k in SCENES} if H == 1000 and SPP == 64 else None
    except Exception:
        return None


def host_cpu_quota():
    """CPUs this container may actually use (cgroup v2 cpu.max), or None when unlimited/unknown."""
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        return None if quota == "max" else round(int(quota) / int(period), 2)
    except Exception:
        pass
    try:  # cgroup v1
        quota = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
        period = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
        return None if quota <= 0 else round(quota / period, 2)
    except Exception:
        return None


def ncu_issue_counters():
    """Issue-side counters of the committed ncu captures of the default kernel (profiles/issue_counters.json)."""
    try:
        with open(os.path.join(ROOT, "profiles", "issue_counters.json")) as f:
            return json.load(f)
    except Exception:
        return None


def measured_peak_gbs():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """Samples SM clocks and throttle reasons during the timed region (pynvml; nvidia-smi as a fallback)."""

    def __init__(self, index=0, period=0.1):
        self.index, self.period = index, period
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thr = None
        self._nvml = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nvml = pynvml
            self._h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self._nvml = None
        self._thr = threading.Thread(target=self._run, daemon=True)
        self._thr.start()

    def _run(self):
        names = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
                 0x80: "hw_power_brake_slowdown", 0x2: "applications_clocks_setting", 0x100: "display_clock_setting"}
        while not self._stop.is_set():
            try:
                if self._nvml:
                    self.samples.append(self._nvml.nvmlDeviceGetClockInfo(self._h, self._nvml.NVML_CLOCK_SM))
                    try:
                        mask = self._nvml.nvmlDeviceGetCurrentClocksEventReasons(self._h)
                    except Exception:
                        mask = self._nvml.nvmlDeviceGetCurrentClocksThrottleReasons(self._h)
                    for bit, nm in names.items():
                        if mask & bit:
                            self.reasons.add(nm)
                else:
                    import subprocess
                    out = subprocess.run(["nvidia-smi", f"--id={self.index}", "--query-gpu=clocks.sm,clocks.max.sm",
                                          "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                    a, b = out.strip().split(",")
                    self.samples.append(int(a))
                    self.max_mhz = int(b)
            except Exception:
                pass
            self._stop.wait(self.period)

    def stop(self):
        self._stop.set()
        if self._thr:
            self._thr.join(timeout=2)
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


# ------------------------------------------------------------------------------------------ CPU legs
def cpu_sample(threads=0, keep=None):
    """Times the oracle on rows j % ROW_STEP == 0 of both headline frames at SPP.  Returns
    (segments, seconds, cores); with `keep` (a dict) the sampled frames are stored in it per scene, so the
    GPU leg can compare the same rows of its own frames (the parity block of the JSON line)."""
    from oracle import pyoracle as O
    if threads <= 0:  # all host threads the container may actually run: the cgroup CPU quota when there is one
        q = host_cpu_quota()
        threads = max(1, int(q + 0.5)) if q else 0
    cores = O.num_procs() if threads <= 0 else threads
    segs, secs = 0, 0.0
    for name in SCENES:
        pr = O.Scene.named(name).prepare(H, W)
        t0 = time.perf_counter()
        pix, _, cnt = pr.render(H, W, spp=SPP, row_start=0, row_step=ROW_STEP, threads=threads)
        secs += time.perf_counter() - t0
        segs += cnt["segments"]
        if keep is not None:
            keep[name] = pix
    return segs, secs, cores


def rows_differing(gpu_frame, oracle_frame, row_start, row_step):
    """(#rows, #pixels, #differing pixels) between a GPU frame and the oracle's row sample of the same frame."""
    import numpy as np
    rows = np.arange(row_start, gpu_frame.shape[0], row_step)
    g, w = np.asarray(gpu_frame)[rows], np.asarray(oracle_frame)[rows]
    return int(rows.size), int(g.size), int((g != w).sum())


# Useful-instruction model of the "issue" roofline: the fewest SASS thread-instructions one aabb_hit / one sphere_hit of
# the reference needs on sm_100a with bit-exact f32 (no FMA contraction): 6 FADD + 6 FMUL + 6 FSEL + 4 FMNMX3/FMNMX +
# 1 FSETP per box (the three reciprocals are per segment); oc (3 FADD), b and c (7 FMUL + 5 FADD), disc (2 FMUL + 1 FADD),
# 1 FSETP + the amortised sqrt / divide / range checks of the ~45 % of tests with disc > 0 for a sphere.
MIN_BOX_INSTR = 23
MIN_SPHERE_INSTR = 30
PUBLISHED_1SPP_MS = {"futhark_multicore_ryzen1700x": {"rgbbox": 179, "irreg": 62}, "futhark_gpu_mi100": {"rgbbox": 14, "irreg": 8}}


def full_frame_equals_oracle(frame, key):
    """True / False: SHA-256 of a whole frame (int32[h][w]) against the oracle's known answer `key` of
    tests/golden/oracle_frame_hashes.json (tools/make_oracle_hashes.py); None when no answer is recorded for that config."""
    import hashlib
    import numpy as np
    with open(os.path.join(ROOT, "tests", "golden", "oracle_frame_hashes.json")) as f:
        known = json.load(f).get(key)
    if not known:
        return None
    return hashlib.sha256(np.ascontiguousarray(frame, "<i4").tobytes()).hexdigest() == known["sha256_le_i32"]


DUMP_BYTES = 48 * 10**6   # all arrays --dump-outputs writes together


def dump_outputs(out_dir, frames):
    """--dump-outputs: every int32[h][w] frame of `frames` as out_dir/<name>.npy in float64 (exact for every int32).  When
    the frames would take more than DUMP_BYTES, each is written as a 1-D array of its pixels at a fixed sample of row-major
    positions (seed 0, ascending), the same positions in every run."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    cap = DUMP_BYTES // (8 * len(frames))
    for name, frame in frames.items():
        out = np.asarray(frame).astype(np.float64)
        if out.size > cap:
            out = out.reshape(-1)[np.sort(np.random.default_rng(0).choice(out.size, cap, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), out)


def issue_roofline(work, ms, sm_count, sm_mhz):
    """Instruction-issue roofline of a render launch: useful thread-instructions of the REFERENCE traversal's box and
    sphere tests / (SMs x 4 schedulers x 32 lanes x clock x time).  This, not HBM, is what bounds the kernel."""
    useful = MIN_BOX_INSTR * work["box_tests"] + MIN_SPHERE_INSTR * work["leaf_tests"]
    peak = sm_count * 4 * 32 * sm_mhz * 1e6            # thread-instructions per second
    ach = useful / (ms * 1e-3)
    return {"bound": "issue", "achieved": round(ach / 1e12, 3), "peak": round(peak / 1e12, 3), "unit": "T thread-instr/s",
            "frac": round(ach / peak, 4), "useful_thread_instr": useful}


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path on this box's host cores.
    The Futhark compiler is not in the image (and its generated ray.c is not in the reference tree), so
    this is the oracle port (bit-exact vs the reference's golden images), all host threads."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    for _ in range(args.warmup):
        cpu_sample()
    segs = secs = 0.0
    cores = 1
    kept = {}
    t_all = time.perf_counter()
    for _ in range(args.steps):
        s, t, cores = cpu_sample(keep=kept)
        segs += s
        secs += t
    wall = time.perf_counter() - t_all
    if args.dump_outputs:   # the last step's frames: the sampled rows, zeros elsewhere
        dump_outputs(args.dump_outputs, kept)
    value = segs / secs / 1e6
    sample = f"rows j%{ROW_STEP}==0 of every {W}x{H} frame of the step at {SPP} spp (1/{ROW_STEP} of a step) per step"
    line = {
        "impl": "reference", "metric": METRIC, "value": round(value, 3), "unit": "Mrays/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(1e3 * wall / args.steps, 3),
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "sample": sample, "host": "cpu"},
        "cpu_baseline": {"value": round(value, 3), "unit": "Mrays/s", "cores": cores, "cgroup_cpu_quota": host_cpu_quota(),
                         "kind": "port", "sample": sample, "per_core": round(value / max(cores, 1), 3),
                         "sample_bias": ({"segments_in_sample_x_row_step": int(segs / args.steps) * ROW_STEP, "segments_per_step": FULL_STEP_SEGMENTS[args.workload],
                                          "ratio": round(segs / args.steps * ROW_STEP / FULL_STEP_SEGMENTS[args.workload], 4)}
                                         if args.workload in FULL_STEP_SEGMENTS else None),
                         "note": "oracle = bit-exact C++ port of the Futhark program (no Futhark compiler in the image); the reference README's "
                                 "Futhark multicore numbers (1 spp 1000x1000, Ryzen 1700X, 8 cores): 179 ms rgbbox / 62 ms irreg = 22.5 / 27.9 Mrays/s"},
        "e2e": {"value": round(value, 3), "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


# ------------------------------------------------------------------------------------------ GPU leg
def run_ours(args):
    import numpy as np
    import torch

    import raytracers_b200 as R
    from raytracers_b200 import distributed as D

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    if args.dump_outputs and world > 1:
        raise SystemExit("--dump-outputs needs --gpus 1")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the product has no CPU path; use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    ctx = R.Context(device=local_rank, kernel=args.kernel)
    stream = torch.cuda.Stream()          # one stream for the library's kernels, NCCL and the timing events
    torch.cuda.set_stream(stream)
    ctx.set_stream(stream.cuda_stream)
    prepared = {name: ctx.prepare_scene(H, W, ctx.scene(name)) for name in SCENES}
    ctx.sync()

    # work per frame (untimed): the counting kernel visits exactly the reference's boxes and leaves
    work = {name: ctx.count_work(H, W, prepared[name], spp=SPP) for name in SCENES} if rank == 0 else None
    if dist is not None:
        box = [work]
        dist.broadcast_object_list(box, src=0)
        work = box[0]
    seg_per_step = sum(work[n]["segments"] for n in SCENES)
    alg_bytes = {n: 32 * work[n]["box_tests"] + 16 * work[n]["leaf_tests"] + 4 * H * W for n in SCENES}

    frames = {n: torch.empty((H, W), dtype=torch.int32, device="cuda") for n in SCENES}
    # N > 1: "peer" = every rank's kernel writes its pixels straight into rank 0's frame over NVLink (the gather fused into
    # the render kernel, D.PeerFrameRenderer); "nccl" = compact tile buffers + one NCCL gather + de-tiling kernel per frame
    sharded = D.ShardedRenderer(ctx, rank, world) if world > 1 else None
    peer = D.PeerFrameRenderer(ctx, rank, world, H, W, slots=4) if world > 1 and args.gather == "peer" else None
    flush = torch.empty(160 * 1024 * 1024, dtype=torch.uint8, device="cuda")  # > 126 MB L2

    # One step = every frame of the workload, submitted as ONE batch (ray_b200_render_batch: two frames in flight, so
    # the long-path tail of a frame is covered by the start of the next); the frame with the longest tail goes first.
    order = sorted(SCENES, key=lambda n: n != "irreg")

    def step():
        if args.no_batch:
            for name in SCENES:
                if sharded is None:
                    ctx.render_into(frames[name].data_ptr(), H, W, prepared[name], spp=SPP)
                else:
                    sharded.render(H, W, prepared[name], spp=SPP)
        elif sharded is None:
            ctx.render_batch([dict(prepared=prepared[n], h=H, w=W, spp=SPP, out_dev=frames[n].data_ptr()) for n in order])
        elif peer is not None:
            peer.render([(prepared[n], SPP) for n in order])
            if rank == 0:   # the step ends when every rank's pixels of its frames have landed in rank 0's HBM
                stream.wait_event(peer.landed)
        else:
            sharded.render_batch([(H, W, prepared[n], SPP) for n in order])

    def strict_steps(k_steps):
        """Round-1 protocol: every step is one JOINED batch between its own event pair, L2 flush outside the pairs."""
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(k_steps)]
        for k in range(k_steps):
            flush.zero_()            # L2 flush between timed steps (untimed: outside the event pair)
            evs[k][0].record(stream)
            step()
            evs[k][1].record(stream)
        barrier()
        return sum(a.elapsed_time(b) for a, b in evs)

    def pipelined_steps(k_steps):
        """K steps submitted back to back with pipelined submission (ray_b200_context_set_pipeline): frames alternate between
        the context's two lanes ACROSS steps, so a frame's last 50-bounce paths are covered by the next frame's start
        instead of idling the GPU at every step boundary.  ONE event pair around all K steps; the per-step L2 flush runs
        inside it (on the context's stream, i.e. between the lane-0 frames of consecutive steps)."""
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ctx.set_pipeline(True)
        e0.record(stream)
        for k in range(k_steps):
            flush.zero_()
            if peer is not None:
                peer.render([(prepared[n], SPP) for n in order])
            else:
                ctx.render_batch([dict(prepared=prepared[n], h=H, w=W, spp=SPP, out_dev=frames[n].data_ptr()) for n in order])
        ctx.pipeline_join()
        if peer is not None and rank == 0:   # ... and every rank's pixels of the last frames have landed in rank 0's HBM
            stream.wait_event(peer.landed)
        e1.record(stream)
        barrier()
        if peer is not None:
            peer.wait()
        ctx.set_pipeline(False)
        return e0.elapsed_time(e1)

    can_pipeline = not args.no_batch and not args.strict_steps and (world == 1 or peer is not None)
    for _ in range(max(args.warmup, 3)):
        step()
    if can_pipeline:
        pipelined_steps(2)
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = ctx.launch_count()
    barrier()
    dev_ms = pipelined_steps(args.steps) if can_pipeline else strict_steps(args.steps)
    launches = ctx.launch_count() - launches0
    clocks = sampler.stop() if rank == 0 else None
    t = torch.tensor([dev_ms], dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms = float(t.item())
    if args.dump_outputs:   # the frames of the last timed step, before the passes below render into the same buffers
        dump_outputs(args.dump_outputs, {n: frames[n].cpu().numpy() for n in SCENES})
    value = seg_per_step * args.steps / (dev_ms * 1e-3) / 1e6
    strict = None
    if can_pipeline:   # the same K steps in the round-1 protocol, for comparison
        barrier()
        ts = torch.tensor([strict_steps(args.steps)], dtype=torch.float64, device="cuda")
        if dist is not None:
            dist.all_reduce(ts, op=dist.ReduceOp.MAX)
        strict = {"value": round(seg_per_step * args.steps / (float(ts.item()) * 1e-3) / 1e6, 1), "ms_per_step": round(float(ts.item()) / args.steps, 4),
                  "protocol": "every step one joined batch between its own event pair, L2 flush outside the pairs (round-1 protocol)"}

    # per-kernel durations for the roofline (N=1: one persistent launch per frame), CUDA events on the launch stream
    roof = issue_all = None
    per_scene = {}
    if rank == 0 and world == 1:
        for name in SCENES:
            ms = []
            for _ in range(5):
                flush.zero_()
                ctx.render_into(frames[name].data_ptr(), H, W, prepared[name], spp=SPP)
                torch.cuda.synchronize()
                ms.append(ctx.last_render_ms())
            ms.sort()
            per_scene[name] = {"ms_per_frame": round(ms[len(ms) // 2], 4), "segments": work[name]["segments"],
                               "Mrays_s": round(work[name]["segments"] / ms[len(ms) // 2] / 1e3, 1),
                               "algorithmic_GB": round(alg_bytes[name] / 1e9, 3),
                               "GB_s": round(alg_bytes[name] / ms[len(ms) // 2] / 1e6, 1)}
        peak, how = measured_peak_gbs()
        tot_bytes = sum(alg_bytes.values())
        tot_ms = sum(per_scene[n]["ms_per_frame"] for n in SCENES)
        ach = tot_bytes / tot_ms / 1e6
        traffic = dram_traffic_per_launch()
        sm_count = torch.cuda.get_device_properties(local_rank).multi_processor_count
        sm_mhz = (clocks or {}).get("sm_mhz") or (clocks or {}).get("sm_max_mhz") or 1965
        work_spp = {n: {k: work[n][k] for k in ("box_tests", "leaf_tests")} for n in SCENES}
        issue = {n: issue_roofline(work_spp[n], per_scene[n]["ms_per_frame"], sm_count, sm_mhz) for n in SCENES}
        tot_useful = sum(issue[n]["useful_thread_instr"] for n in SCENES)
        issue_all = {"bound": "issue", "achieved": round(tot_useful / (tot_ms * 1e-3) / 1e12, 3), "peak": issue[SCENES[0]]["peak"],
                     "unit": "T thread-instr/s", "frac": round(tot_useful / (tot_ms * 1e-3) / (issue[SCENES[0]]["peak"] * 1e12), 4),
                     "per_scene": {n: issue[n]["frac"] for n in SCENES}, "sm_mhz": sm_mhz, "sm_count": sm_count,
                     "model": f"useful = {MIN_BOX_INSTR} thread-instr x box tests + {MIN_SPHERE_INSTR} x sphere tests of the REFERENCE "
                              "traversal (bit-exact f32, no FMA); peak = SMs x 4 schedulers x 32 lanes x SM clock",
                     "ncu": ncu_issue_counters()}
        roof = {"bound": "hbm", "achieved": round(ach, 1), "peak": peak, "unit": "GB/s", "frac": round(ach / peak, 4),
                "traffic": (sum(traffic.values()) / len(traffic) if traffic else None), "traffic_per_scene": traffic,
                "traffic_source": "profiles/dram_traffic.json (ncu --set full, per launch)", "peak_source": how, "kernel": f"render ({args.kernel}) — one launch per frame",
                "algorithmic_bytes_per_launch": {n: alg_bytes[n] for n in SCENES}, "per_scene": per_scene,
                "note": "ACCOUNTING figure, not a bound: algorithmic bytes = 32 B x box tests + 16 B x sphere tests of the REFERENCE "
                        "traversal + 4 B x pixels (SURVEY 8d) relative to the HBM copy peak; the scene (<1 MB) is shared-memory/L2 "
                        "resident, real DRAM traffic is `traffic`, so the fraction can exceed 1 - the kernel is bound by "
                        "instruction issue and shared-memory bandwidth: see roofline_issue"}

    # N > 1 diagnostic: this rank's render-kernel time per frame (shard only, no gather), to separate kernel scaling
    # from collective / synchronisation cost
    rank_kernel_ms = None
    if world > 1:
        mine = {}
        shard_tiles, _ = sharded._buffers(H, W)
        for name in SCENES:
            ms = []
            for _ in range(5):
                ctx.render_shard_into(shard_tiles.data_ptr(), H, W, prepared[name], spp=SPP)
                torch.cuda.synchronize()
                ms.append(ctx.last_render_ms())
            mine[name] = round(sorted(ms)[2], 3)
        allv = [None] * world
        dist.all_gather_object(allv, mine)
        rank_kernel_ms = {n: [v[n] for v in allv] for n in SCENES}

    # e2e: host buffers through the public API; per step, inside the timed region (wall clock, barrier + synchronize on both
    # sides): H2D of every scene's sphere records from page-locked memory + device LBVH build (on every rank), all frames of
    # the step as one batch, and every frame's D2H into page-locked host memory (rank 0).
    #   default ("peer", also at N = 1): D.PeerFrameRenderer with pipelined submission - the frames land in rank 0's ring
    #     (over NVLink from the other ranks) and are copied out on its copy stream while the next frames render; nothing
    #     blocks the host but the re-upload's own 32-byte read-back;
    #   --gather nccl (N > 1): tile buffers + ncclGather + de-tile per frame, D2H on a second stream ordered by events;
    #   --strict-steps / --no-batch at N = 1: the round-1 loop (futhark_entry_render-style call, blocking futhark_values).
    e2e = None
    h2d = sum(prepared[n].upload_bytes() for n in SCENES)
    d2h = 4 * H * W * len(SCENES)
    e2e_how = None
    if can_pipeline:
        e2e_how = "peer-frame ring + pipelined submission"
        pf = peer if peer is not None else D.PeerFrameRenderer(ctx, rank, world, H, W, slots=4)
        ctx.set_pipeline(True)

        def e2e_steps(n_steps):
            for _ in range(n_steps):
                for name in SCENES:
                    prepared[name].reupload()                       # H2D from pinned memory + LBVH build on the device
                pf.render([(prepared[n], SPP) for n in order])      # render + (rank 0) flag wait, D2H, slot release on the copy stream
            pf.wait()                                               # every frame of every step is in host memory

        e2e_steps(2)
        barrier()
        t0 = time.perf_counter()
        e2e_steps(args.steps)
        barrier()
        e2e_s = time.perf_counter() - t0
        ctx.set_pipeline(False)
        if rank == 0 and not args.no_cpu_baseline:   # the frames that reached the host are the frames the kernels wrote
            got = {n: pf.host[(pf.seq - len(order) + i) % pf.slots].numpy().copy() for i, n in enumerate(order)}
        else:
            got = None
        if peer is None:
            pf.close()
    elif world == 1:
        e2e_how = "futhark_entry_render-style call per frame, blocking futhark_values_i32_2d"
        got = None
        host = {n: torch.empty((H, W), dtype=torch.int32, pin_memory=True) for n in SCENES}

        def e2e_step():
            for name in SCENES:
                prepared[name].reupload()                                   # H2D of the sphere records from pinned memory + device LBVH build
                img = ctx.render(H, W, prepared[name], spp=SPP)             # futhark_entry_render-style call
                ctx.lib.futhark_values_i32_2d(ctx.handle, img.handle, host[name].data_ptr())  # D2H + sync (main.c:130)
                img.free()

        for _ in range(2):
            e2e_step()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            e2e_step()
        torch.cuda.synchronize()
        e2e_s = time.perf_counter() - t0
    else:
        e2e_how = "NCCL gather + de-tile per frame, D2H on a copy stream"
        got = None
        host = [torch.empty((H, W), dtype=torch.int32, pin_memory=True) for _ in SCENES] if rank == 0 else None
        copy_stream = torch.cuda.Stream() if rank == 0 else None
        copied = [torch.cuda.Event() for _ in SCENES] if copy_stream is not None else None
        barrier()
        t0 = time.perf_counter()
        for k in range(args.steps):
            for name in SCENES:
                prepared[name].reupload()
            if copied is not None and k > 0:
                for ev_c in copied:          # the frame buffers are reused: last step's copies must have read them
                    stream.wait_event(ev_c)
            frs = sharded.render_batch([(H, W, prepared[n], SPP) for n in order])
            if rank == 0:
                ready_ev = torch.cuda.Event()
                ready_ev.record(stream)
                copy_stream.wait_event(ready_ev)
                with torch.cuda.stream(copy_stream):
                    for i, fr in enumerate(frs):
                        host[i].copy_(fr, non_blocking=True)
                        copied[i].record(copy_stream)
        if copy_stream is not None:
            copy_stream.synchronize()
        barrier()
        e2e_s = time.perf_counter() - t0
    tt = torch.tensor([e2e_s], dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    e2e = {"value": round(seg_per_step * args.steps / float(tt.item()) / 1e6, 1), "unit": "Mrays/s", "h2d_bytes_per_step": h2d,
           "d2h_bytes_per_step": d2h, "ms_per_step": round(1e3 * float(tt.item()) / args.steps, 3), "how": e2e_how}

    # context: the reference's own published protocol (1 sample per pixel, README table) on this GPU
    one_spp = None
    if rank == 0 and world == 1:
        one_spp = {}
        for name in (SCENES if H <= 2000 else ()):
            ms = []
            for _ in range(7):
                ctx.render_into(frames[name].data_ptr(), H, W, prepared[name], spp=1)
                torch.cuda.synchronize()
                ms.append(ctx.last_render_ms())
            ms.sort()
            one_spp[name] = round(ms[len(ms) // 2], 4)
        if one_spp:   # the same two fractions for the reference's own 1-ray-per-pixel protocol (README.md:43-51, main.c:107-120)
            peak, _ = measured_peak_gbs()
            smc = torch.cuda.get_device_properties(local_rank).multi_processor_count
            frac = {}
            for name in list(one_spp):
                wk1 = ctx.count_work(H, W, prepared[name], spp=1)
                gb = (32 * wk1["box_tests"] + 16 * wk1["leaf_tests"] + 4 * H * W) / 1e9
                frac[name] = {"hbm_accounting_frac": round(gb / one_spp[name] * 1e3 / peak, 4),
                              "issue_frac": issue_roofline(wk1, one_spp[name], smc, (clocks or {}).get("sm_mhz") or 1965)["frac"],
                              "Mrays_s": round(wk1["segments"] / one_spp[name] / 1e3, 1)}
            one_spp["fractions"] = frac

    # The other BASELINE configs (north-star target sizes), once each outside the timed steps: irreg 4000x4000 at 1 and
    # 256 spp (configs[3]) and the 1 M-sphere scene (configs[4]), each with an oracle row-sample parity check.
    extra = None
    if rank == 0 and world == 1 and not args.no_extra:
        from oracle import pyoracle as O
        extra = {}
        peak, _ = measured_peak_gbs()
        sm_count = torch.cuda.get_device_properties(local_rank).multi_processor_count
        sm_mhz = (clocks or {}).get("sm_mhz") or 1965
        threads = max(1, int((host_cpu_quota() or 0) + 0.5)) or 0
        for tag, scene_args, hh, ww, spp, row_start, row_step in (
                ("irreg_4000x4000_1spp", ("irreg",), 4000, 4000, 1, 0, 4),
                ("irreg_4000x4000_256spp", ("irreg",), 4000, 4000, 256, 128, 512),
                ("random1M_2000x2000_16spp", ("random", 1000000, 1), 2000, 2000, 16, 125, 500)):
            t0 = time.perf_counter()
            sc = ctx.scene(scene_args[0], n=scene_args[1] if len(scene_args) > 1 else None)
            pr = ctx.prepare_scene(hh, ww, sc)
            ctx.sync()
            prep_s = time.perf_counter() - t0
            wk = ctx.count_work(hh, ww, pr, spp=spp)
            fr = torch.empty((hh, ww), dtype=torch.int32, device="cuda")
            ms = []
            for _ in range(3 if spp * hh * ww < 2e9 else 2):
                ctx.render_into(fr.data_ptr(), hh, ww, pr, spp=spp)
                torch.cuda.synchronize()
                ms.append(ctx.last_render_ms())
            m = sorted(ms)[(len(ms) - 1) // 2]   # (lower) median; the first frame of a scene also records the learned claim order
            gb = (32 * wk["box_tests"] + 16 * wk["leaf_tests"] + 4 * hh * ww) / 1e9
            par = None
            if not args.no_cpu_baseline:   # oracle rows (j - row_start) % row_step == 0 of this very frame
                o_sc = O.Scene.named(scene_args[0], **({"n": scene_args[1], "seed": scene_args[2]} if len(scene_args) > 1 else {}))
                t0 = time.perf_counter()
                want, _, ocnt = o_sc.prepare(hh, ww).render(hh, ww, spp=spp, row_start=row_start, row_step=row_step, threads=threads)
                fr_host = fr.cpu().numpy()
                rows, pixels, bad = rows_differing(fr_host, want, row_start, row_step)
                par = {"rows": rows, "pixels": pixels, "differing": bad, "oracle_segments": ocnt["segments"],
                       "oracle_s": round(time.perf_counter() - t0, 2)}
                try:   # every pixel: SHA-256 of the whole frame against the oracle's known answer for this config (never fatal)
                    same = full_frame_equals_oracle(fr_host, tag)
                    if same is not None:
                        par["full_frame_sha256_equals_oracle"] = same
                except Exception as e:  # noqa: BLE001
                    print(f"bench: full-frame known-answer check of {tag} skipped: {e}", file=sys.stderr)
                del fr_host
            extra[tag] = {"ms_per_frame": round(m, 3), "segments": wk["segments"], "Mrays_s": round(wk["segments"] / m / 1e3, 1),
                          "algorithmic_GB": round(gb, 2), "GB_s": round(gb / m * 1e3, 1), "roofline_frac": round(gb / m * 1e3 / peak, 4),
                          "issue_frac": issue_roofline(wk, m, sm_count, sm_mhz)["frac"], "parity": par,
                          "prepare_scene_s": round(prep_s, 3), "info": {k: (int(v) if not hasattr(v, "shape") else None) for k, v in pr.info().items() if k in ("n_leaves", "max_depth", "smem_nodes", "stale_nodes")}}
            del fr
            pr.free(); sc.free()

    cpu = parity = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        kept = {}
        segs, secs, cores = cpu_sample(keep=kept)
        rate = segs / secs / 1e6
        cpu = {"value": round(rate, 3), "unit": "Mrays/s", "cores": cores, "cgroup_cpu_quota": host_cpu_quota(), "kind": "port",
               "per_core": round(rate / cores, 3),
               "sample": f"rows j%{ROW_STEP}==0 of every {W}x{H} frame of the step at {SPP} spp (1/{ROW_STEP} of a step), {secs:.1f} s",
               "sample_bias": {"segments_in_sample_x_row_step": segs * ROW_STEP, "segments_per_step": seg_per_step,
                               "ratio": round(segs * ROW_STEP / seg_per_step, 4)},
               "note": "oracle = bit-exact C++ port of the Futhark program (the Futhark compiler is not in the image); the "
                       "reference README's own Futhark multicore numbers (1 spp 1000x1000, Ryzen 1700X, 8 cores) are "
                       "179 ms rgbbox / 62 ms irreg = 22.5 / 27.9 Mrays/s, i.e. ~3 Mrays/s per core - a GPU/CPU ratio "
                       "against this port is NOT a ratio against Futhark on this host"}
        # parity of the timed workload itself: the same rows of the GPU frames the timed steps produced
        parity = {"vs": "oracle (CPU port, bit-exact vs the reference's golden PNGs)", "kernel": args.kernel, "scenes": {}}
        for name in SCENES:
            ctx.render_into(frames[name].data_ptr(), H, W, prepared[name], spp=SPP)
            torch.cuda.synchronize()
            rows, pixels, bad = rows_differing(frames[name].cpu().numpy(), kept[name], 0, ROW_STEP)
            parity["scenes"][name] = {"rows": rows, "pixels": pixels, "differing": bad}
        if got is not None:   # ... and the frames the e2e leg delivered to HOST memory (through the peer-frame ring)
            for name in SCENES:
                rows, pixels, bad = rows_differing(got[name], kept[name], 0, ROW_STEP)
                parity["scenes"][name]["e2e_host_frame_differing"] = bad
        parity["differing"] = sum(v["differing"] + v.get("e2e_host_frame_differing", 0) for v in parity["scenes"].values())

    if rank == 0 and got is not None:
        # every pixel of the frames the end-to-end leg delivered to host memory (at N > 1: assembled from all ranks' stores)
        # against the oracle's known answers for these frames (tests/golden/oracle_frame_hashes.json); never fatal
        try:
            full = {n: full_frame_equals_oracle(got[n], f"{n}_{H}x{W}_{SPP}spp") for n in SCENES}
            full = {n: v for n, v in full.items() if v is not None}
            if full:
                if parity is None:
                    parity = {"vs": "SHA-256 of the oracle's full frames (tests/golden/oracle_frame_hashes.json)", "scenes": {}}
                for n in full:
                    parity["scenes"].setdefault(n, {})["e2e_host_frame_sha256_equals_oracle_full_frame"] = full[n]
                parity["differing_frames"] = sum(not v for v in full.values())
        except Exception as e:  # noqa: BLE001
            print(f"bench: full-frame known-answer check skipped: {e}", file=sys.stderr)

    if rank == 0:
        line = {
            "metric": METRIC, "value": round(value, 1), "unit": "Mrays/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": round(dev_ms / args.steps, 4), "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "kernel": args.kernel, "spp": SPP, "segments_per_step": seg_per_step,
                       "l2": ("flushed every step (160 MiB memset on the context's stream, inside the single event pair of the K pipelined steps); scene is <1 MB"
                              if can_pipeline else "flushed between timed steps (160 MiB memset outside the event pairs); scene is <1 MB"),
                       "timing": ("K steps submitted back to back with pipelined submission (frames alternate between two lanes across steps), one CUDA-event pair around all K steps"
                                  if can_pipeline else "one CUDA-event pair per step (joined batch)"),
                       "parallelism": (f"tile-sharded x{world}, " + ("pixels written straight into rank 0's frame over NVLink peer memory (gather fused into the render kernel)"
                                                                      if args.gather == "peer" else "one NCCL gather per frame")) if world > 1 else "single GPU",
                       "submission": "frame by frame" if args.no_batch else "one ray_b200_render_batch per step (two frames in flight)",
                       "ray": "one ray segment = one objs_hit call (ray.fut:76-86)"},
            "strict_steps": strict, "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks, "roofline": roof, "roofline_issue": issue_all,
            "parity": parity, "cpu_baseline": cpu,
            "frame_ms_1spp": one_spp, "learned_claim_order": os.environ.get("RAY_LEARN_ORDER", "1") != "0", "extra": extra, "shard_kernel_ms_per_rank": rank_kernel_ms,
            "published_reference_1spp_ms": PUBLISHED_1SPP_MS,
        }
        print(json.dumps(line), flush=True)
    if peer is not None:
        dist.barrier()
        peer.close()
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    return 0


# segments of one full step (GPU counting kernel = the oracle's bvh_fold counters, tests/test_gpu_parity.py): lets the CPU arm
# show that its row sample is unbiased without rendering the other 7/8 of the step
FULL_STEP_SEGMENTS = {"headline": 368008372, "irreg4000": 7081424953}

WORKLOADS = {
    # name: (scenes, H, W, spp, metric, workload description, rows the CPU legs sample)
    "headline": (("rgbbox", "irreg"), 1000, 1000, 64, "Mrays/s (ray segments/s) rgbbox+irreg 1000x1000",
                 "rgbbox 1000x1000 64spp + irreg 1000x1000 64spp per step (BASELINE.json configs[1]+configs[2])", 8),
    "irreg4000": (("irreg",), 4000, 4000, 256, "Mrays/s (ray segments/s) irreg 4000x4000 256spp",
                  "irreg 4000x4000 256spp per step (BASELINE.json configs[3])", 512),
}


def select_workload(name):
    global SCENES, H, W, SPP, METRIC, WORKLOAD, ROW_STEP
    SCENES, H, W, SPP, METRIC, WORKLOAD, ROW_STEP = WORKLOADS[name]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--kernel", default=os.environ.get("RAY_KERNEL", "auto"))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-batch", action="store_true", help="submit the frames of a step one by one instead of as one batch")
    ap.add_argument("--strict-steps", action="store_true", help="time every step as one joined batch between its own event pair (round-1 protocol) instead of K pipelined steps")
    ap.add_argument("--no-extra", action="store_true",
                    help="skip the once-per-run measurement (outside the timed steps) of BASELINE configs[3] and [4]: irreg 4000x4000 at 1 / 256 spp and the 1M-sphere scene")
    ap.add_argument("--extra", action="store_true", help="(default now; kept for compatibility)")
    ap.add_argument("--gather", default=os.environ.get("RAY_GATHER", "peer"), choices=["peer", "nccl"],
                    help="N > 1: peer = ranks write their pixels straight into rank 0's frame over NVLink (default); nccl = tile buffers + ncclGather + de-tile")
    ap.add_argument("--workload", default="headline", choices=sorted(WORKLOADS),
                    help="headline = BASELINE configs[1]+[2] (the default the driver measures); irreg4000 = configs[3]")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the frames of the last step as DIR/<scene>.npy (float64 packed 0x00RRGGBB "
                         "pixels, a fixed sample of them for frames beyond 48 MB in all; the scenes are fixed, so the same "
                         "arguments give the same inputs in every run)")
    args = ap.parse_args()
    select_workload(args.workload)
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
