#!/usr/bin/env python
"""bench.py — headline benchmark of the PathTrace hot path (BASELINE.json: "Mrays/s and ms/frame @1080p 4spp 6-bounce Bistro").

  python bench.py --gpus N --steps K --warmup W            product arm (CUDA wavefront through the C ABI)
      [--dump-outputs DIR]                                 ... and write the frame the last timed step produced to DIR/accumulated.npy
  python bench.py --impl reference --gpus N ...            reference arm: the reference's algorithm for this path on the host cores
                                                           (RTXPT itself has no CPU implementation and cannot run here — HLSL/DXR, Windows
                                                           only, SURVEY.md F1-F3 — so this arm times the CPU restatement in oracle/)

Workload (configs[1] of BASELINE.json, fits one GPU): 1920x1080, 4 sub-samples per frame, BounceCount 6 / DiffuseBounceCount 6, StandardBSDF,
NEE with 5 candidates + 1 shadow ray per vertex, Russian roulette, firefly filter on, environment map on, on the ~2.8 M triangle procedural
"city block" stand-in for Bistro exterior (the real Bistro assets are git-LFS stubs in the reference tree: SURVEY.md F7).
A step is one frame: 4 sub-samples path traced and folded into the accumulation buffer.  A ray is one traversal query (scatter or shadow).
One JSON line on stdout (rank 0).  The scene is generated from fixed seeds and frame i uses sample indices 4i..4i+3, so the same arguments give the
same inputs on every run; the benchmark writes nothing into the source tree (the tree may be read-only).
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.dont_write_bytecode = True          # no __pycache__ in the tree

import numpy as np

WIDTH, HEIGHT, SPP, BOUNCES = 1920, 1080, 4, 6
TARGET_TRIANGLES = 2_800_000
FIREFLY_THRESHOLD = 5000.0          # ReferenceFireflyFilterThreshold 5 * sqrt(preExposedGray = 1) * 1e3 (Rtxpt/Sample.cpp:1522, SampleUI.h:212-213)


def build_workload(width=WIDTH, height=HEIGHT, triangles=TARGET_TRIANGLES):
    from rtxpt_b200 import scenes, scene_builder as sb
    scene, cam = scenes.city_block(target_triangles=triangles, width=width, height=height)
    consts = sb.make_constants(width, height, cam, bounce_count=BOUNCES, diffuse_bounce_count=BOUNCES, env_enabled=True,
                               firefly_threshold=FIREFLY_THRESHOLD, nee=True, nee_type=2)
    return scene, consts


def workload_config(n_gpus):
    return {"workload": "city-block stand-in for Bistro-exterior (configs[1]): %dx%d, %d spp/frame, BounceCount %d, DiffuseBounceCount %d, StandardBSDF + envmap + NEE(5 candidates, 1 shadow ray) + RR + firefly filter"
                        % (WIDTH, HEIGHT, SPP, BOUNCES, BOUNCES),
            "triangles": TARGET_TRIANGLES, "materials": 254, "image": [WIDTH, HEIGHT], "spp_per_frame": SPP,
            "partition": "1 GPU, whole frame" if n_gpus == 1 else "interleaved 64x64 screen tiles over %d GPUs + NCCL all-gather of radiance tiles" % n_gpus,
            "cache": "working set per frame (path state 664 MB + scene ~400 MB) exceeds the 126 MB L2; no explicit flush"}


def _gpu_uuid(torch, index):
    """NVML enumerates physical GPUs, CUDA the visible ones: match by UUID."""
    try: return "GPU-" + str(torch.cuda.get_device_properties(index).uuid)
    except Exception: return None


class ClockSampler:
    """SM clock, power and clock-event reasons of this rank's GPU sampled DURING the timed region (B200_PROFILING.md clocks line).  NVML in a thread of this process (what
    nvidia-smi itself reads): a looping `nvidia-smi -lms` process needed 70-100+ ms per query on the 8-GPU boxes and held the driver while it enumerated the node - the N=8 timed
    loop of round 1 / early round 2 measured 6.7 ms per frame against 3.6 ms for the same frames with a host synchronize in between, with ONE clock sample taken
    (profiles/r2_history.md section 10).  Falls back to nvidia-smi when NVML cannot be loaded."""
    REASONS = (("hw_slowdown", "HwSlowdown"), ("hw_thermal_slowdown", "HwThermalSlowdown"), ("sw_thermal_slowdown", "SwThermalSlowdown"), ("sw_power_cap", "SwPowerCap"))

    def __init__(self, index, uuid=None, period_s=0.01):
        self.sm, self.mx, self.reasons, self.proc, self.nvml, self.stop_flag, self.lines, self.source = [], [], set(), None, None, False, [], "nvml"
        try:
            import pynvml
            pynvml.nvmlInit(); self.nvml = pynvml
            try: self.handle = pynvml.nvmlDeviceGetHandleByUUID(uuid if isinstance(uuid, bytes) else str(uuid).encode()) if uuid else pynvml.nvmlDeviceGetHandleByIndex(index)
            except Exception: self.handle = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_sm = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM)); self.period = period_s
            self.thread = threading.Thread(target=self._poll, daemon=True); self.thread.start()
            return
        except Exception:
            self.nvml = None
        self.source = "nvidia-smi"
        q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + q, "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _poll(self):
        n = self.nvml
        get = getattr(n, "nvmlDeviceGetCurrentClocksEventReasons", None) or n.nvmlDeviceGetCurrentClocksThrottleReasons
        while not self.stop_flag:
            try:
                self.sm.append(float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM))); self.mx.append(self.max_sm)
                bits = int(get(self.handle))
                for name, suffix in self.REASONS:
                    mask = getattr(n, "nvmlClocksEventReason" + suffix, None) or getattr(n, "nvmlClocksThrottleReason" + suffix, 0)
                    if bits & int(mask): self.reasons.add(name)
            except Exception:
                pass
            time.sleep(self.period)

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.nvml is not None:
            self.stop_flag = True; self.thread.join(1.0)
            return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": max(self.mx) if self.mx else None, "reasons": sorted(self.reasons), "samples": len(self.sm), "source": "nvml"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for l in self.lines:
            f = [x.strip() for x in l.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons), "samples": len(sm), "source": "nvidia-smi"}


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_capture(rays_per_iteration):
    """Counters of k_trace_closest from the committed `ncu --set full` capture (profiles/r2_ncu_full_summary.json, else round 1's): DRAM bytes per frame, the share of issue
    slots in use and the executed thread-instructions per ray.  The capture holds the launches of the first iterations of one frame; byte and instruction totals are scaled to
    the frame by this run's ray counts (same unit as `achieved`: per frame = per launch x launches).  The numbers describe the build the capture was taken from: its commit is
    reported next to them, and a capture older than the kernels goes stale - `traffic_note` says which file was read."""
    here = os.path.dirname(os.path.abspath(__file__))
    for name in ("r2_ncu_full_summary.json", "r1_ncu_full_summary.json"):
        path = os.path.join(here, "profiles", name)
        if not os.path.exists(path):
            continue
        try:
            data = json.load(open(path)); rows_all = data["rows"] if isinstance(data, dict) else data
            rows = [r for r in rows_all if "k_trace_closest" in r["kernel"]]
            captured = sum(r["dram_read_bytes"] + r["dram_write_bytes"] for r in rows)
            frac = sum(rays_per_iteration[:len(rows)]) / max(1, sum(rays_per_iteration))
            rays_captured = sum(rays_per_iteration[:len(rows)])
            ms = sum(r["time_ms"] for r in rows)
            out = {"traffic": captured / frac, "capture_ms": ms, "capture_dram_bytes": captured,
                   # time-weighted over the captured launches (the last bounces are a few microseconds at single-digit utilisation: a plain mean would describe them)
                   "issue_active": float(sum(r["issue_active_pct"] * r["time_ms"] for r in rows) / max(ms, 1e-9)) / 100.0 if "issue_active_pct" in rows[0] else None,
                   "threads_per_inst": float(sum(r["threads_per_inst"] * r["time_ms"] for r in rows) / max(ms, 1e-9)) if "threads_per_inst" in rows[0] else None,
                   "thread_inst_per_ray": (sum(r["warp_insts"] * r["threads_per_inst"] for r in rows) / max(1, rays_captured)) if "warp_insts" in rows[0] else None,
                   "commit": data.get("commit") if isinstance(data, dict) else "round 1 (e38f795 or earlier)",
                   "note": "profiles/%s: %d captured launches = %.0f %% of the frame's scatter rays, scaled to the frame" % (name, len(rows), 100 * frac)}
            return out
        except Exception as e:  # malformed capture: say so instead of guessing
            return {"traffic": None, "note": "capture %s unreadable (%s)" % (name, e)}
    return {"traffic": None, "note": "no ncu capture committed under profiles/"}


def cpu_sample_rect():
    # bounded sample of the same workload: a 960x540 window in the middle of the 1080p frame, 1 sub-sample (~2.4 M rays per step: enough rows to keep
    # every host thread busy, about a second per step on 64 cores)
    w, h = 960, 540
    x0, y0 = (WIDTH - w) // 2, (HEIGHT - h) // 2
    return x0, y0, x0 + w, y0 + h


def physical_cores():
    """Host threads the CPU arm uses: one per physical core the process may run on (SMT siblings only slow the BVH-walking oracle down:
    measured 5.5 Mrays/s on 64 threads vs 3.2 on 128 on the GPU box)."""
    try:
        allowed = os.sched_getaffinity(0); cores = set(); cur = {}
        for line in open("/proc/cpuinfo"):
            if ":" in line:
                k, v = [x.strip() for x in line.split(":", 1)]; cur[k] = v
            elif cur:
                if int(cur.get("processor", -1)) in allowed: cores.add((cur.get("physical id", "0"), cur.get("core id", cur.get("processor"))))
                cur = {}
        return max(1, len(cores)) if cores else max(1, len(allowed))
    except Exception:
        return max(1, os.cpu_count() or 1)


def run_cpu(scene, consts, steps, warmup):
    """Times the oracle (CPU restatement of the reference path, OpenMP over all host cores) on the bounded sample; returns Mrays/s etc."""
    import oracle_lib as ol             # the library build() made; not rebuilt here
    t0 = time.time(); o = ol.Oracle(scene); bvh_s = ol.lib().oracle_bvh_build_seconds(o.h)
    o.set_constants(consts); setup_s = time.time() - t0
    rect = cpu_sample_rect()
    rays, secs, cpu_s, wall_s = 0, 0.0, 0.0, 0.0
    for i in range(warmup + steps):
        t_cpu, t_wall = time.process_time(), time.perf_counter()
        acc, n, last, prim, st = o.render(i, 1, rect=rect, threads=physical_cores())
        if i >= warmup:
            rays += st.scatterRays + st.shadowRays; secs += st.seconds
            cpu_s += time.process_time() - t_cpu; wall_s += time.perf_counter() - t_wall
    threads = st.threads
    paths = (rect[2] - rect[0]) * (rect[3] - rect[1]) * steps
    return {"mrays_s": rays / secs / 1e6, "seconds": secs, "rays": rays, "threads": threads, "bvh_build_s": bvh_s, "setup_s": setup_s,
            "ms_per_step": secs / steps * 1e3, "rays_per_path": rays / paths,
            # user+system CPU seconds of this process over the wall time of the timed steps: how many cores the arm really got (a cgroup quota or a noisy neighbour shows here)
            "cpu_seconds": cpu_s, "wall_seconds": wall_s, "cores_busy": cpu_s / max(wall_s, 1e-9), "host_cpus": os.cpu_count(), "loadavg": list(os.getloadavg()),
            "sample": "%dx%d window at the centre of the %dx%d frame, 1 sub-sample per step, %d steps" % (rect[2] - rect[0], rect[3] - rect[1], WIDTH, HEIGHT, steps)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30, help="timed frames of the headline and end-to-end measurements (and of --impl reference); the CPU baseline "
                                                           "(3 steps) and the realtime child (scripts/bench_realtime.py, 10 frames) keep their own counts")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-realtime", action="store_true", help="skip the realtime-mode (stable planes) timing that runs in a child process after the headline measurement")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the accumulated RGBA float32 frame the last timed step left (what a caller reads back) "
                                                           "to DIR/accumulated.npy, so that two builds can be compared on identical inputs")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to the CUDA arm (--impl b200)")
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    n_gpus = args.gpus

    if args.impl == "reference":
        if rank != 0:
            return 0
        scene, consts = build_workload()
        r = run_cpu(scene, consts, max(1, args.steps), min(args.warmup, 1))
        line = {"impl": "reference", "metric": "Mrays/s", "value": r["mrays_s"], "unit": "Mrays/s", "n_gpus": n_gpus, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32 (fp16 path-state storage)",
                "data": "synthetic", "config": workload_config(n_gpus),
                "cpu_baseline": {"value": r["mrays_s"], "unit": "Mrays/s", "cores": r["threads"], "kind": "port", "sample": r["sample"],
                                 "bvh_build_s": r["bvh_build_s"], "rays_per_path": r["rays_per_path"], "cores_busy": r["cores_busy"], "cpu_seconds": r["cpu_seconds"], "wall_seconds": r["wall_seconds"],
                                 "host_cpus": r["host_cpus"], "loadavg": r["loadavg"]},
                "e2e": {"value": r["mrays_s"], "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "note": "RTXPT has no CPU implementation of this path (HLSL/DXR only); this arm times the CPU restatement of its algorithm (oracle/) on the host cores"}
        print(json.dumps(line)); return 0

    real_stdout = os.dup(1); os.dup2(2, 1)          # libraries that print to fd 1 (NCCL's version banner) must not pollute the one-line contract
    import torch
    from rtxpt_b200 import lib, structs as S
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    scene, consts = build_workload()
    # tuning aid (not a bench mode): RTXPT_BENCH_EMULATE_WORLD=N on one GPU renders rank 0's tile set of an N-GPU job, i.e. what one rank of the strong-scaling run computes per frame
    emulate = int(os.environ.get("RTXPT_BENCH_EMULATE_WORLD", "0")) if world == 1 else 0
    ctx = lib.Context(max_sub_samples_per_launch=SPP, device=local_rank, tile_rank=rank if not emulate else 0, tile_world=world if not emulate else emulate, tile_size=64)
    ctx.upload_scene(scene)
    ctx.set_constants(consts)
    owned, padded = ctx.tile_layout()
    send = gathered = None
    if world > 1:
        send = torch.empty((padded, 4), dtype=torch.float32, device="cuda")
        gathered = torch.empty((world * padded, 4), dtype=torch.float32, device="cuda")
    # all GPU work of the benchmark (wavefront kernels, tile pack/unpack, NCCL) goes to one non-default torch stream; the timing events are
    # recorded on that same stream
    tstream = torch.cuda.Stream()
    torch.cuda.set_stream(tstream)
    stream = tstream.cuda_stream
    host_out = torch.empty((HEIGHT, WIDTH, 4), dtype=torch.float32, pin_memory=True).numpy()      # pinned host frame the e2e leg reads back into

    def frame(i):
        consts.sampleBaseIndex = i * SPP
        ctx.set_constants(consts)
        ctx.path_trace(0, SPP, True, stream)
        if world > 1:
            ctx.pack_owned(send.data_ptr(), stream)
            dist.all_gather_into_tensor(gathered, send)
            ctx.unpack_all(gathered.data_ptr(), stream)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident timing: K frames between CUDA events on the launching stream --------------------------------------------------
    for i in range(args.warmup):
        frame(i)
    barrier()
    sampler = ClockSampler(local_rank, uuid=_gpu_uuid(torch, local_rank)) if rank == 0 else None
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    rays = 0; k_closest = k_shadow = k_shade = k_other = 0.0
    ev0.record()
    for i in range(args.steps):
        frame(args.warmup + i)
        # per-frame ray counts come back with the (already asynchronous) counter copy; reading them syncs, so it is done after the loop for all but the last frame
    ev1.record()
    barrier()
    ms_total = ev0.elapsed_time(ev1)
    st = ctx.stats()                         # last frame's counters; rays per frame vary <0.1% between frames with this workload
    rays_per_frame_local = st.scatterRays + st.shadowRays
    t = torch.tensor([ms_total, float(rays_per_frame_local)], dtype=torch.float64, device="cuda")
    if world > 1:
        tmax = t.clone(); dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        tsum = t.clone(); dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
        ms_total = float(tmax[0]); rays_per_frame = float(tsum[1])
    else:
        rays_per_frame = float(rays_per_frame_local)
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:
        # after the clock sampler (the GPU idles during the file write) and before the e2e leg (which keeps accumulating into the same buffer); rank 0 holds
        # the whole frame (N > 1: after the all-gather of the last step); 1920 x 1080 x 4 float32 = 33 MB
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "accumulated.npy"), ctx.readback_accumulated())
    ms_per_step = ms_total / args.steps
    value = rays_per_frame / (ms_per_step * 1e-3) / 1e6

    # ---- where a frame's time goes on this rank (N > 1: the scaling curve's explanation): CUDA events between the phases of 6 further frames, max over ranks per phase ------
    phases = None
    if world > 1:
        names = ["set_constants+path_trace", "pack", "all_gather", "unpack"]
        acc = np.zeros(len(names)); frames_p = 6
        for i in range(frames_p):
            evs = [torch.cuda.Event(enable_timing=True) for _ in range(len(names) + 1)]
            consts.sampleBaseIndex = (args.warmup + args.steps + i) * SPP
            evs[0].record(); ctx.set_constants(consts); ctx.path_trace(0, SPP, True, stream)
            evs[1].record(); ctx.pack_owned(send.data_ptr(), stream)
            evs[2].record(); dist.all_gather_into_tensor(gathered, send)
            evs[3].record(); ctx.unpack_all(gathered.data_ptr(), stream)
            evs[4].record(); torch.cuda.synchronize()
            if i > 0: acc += np.array([evs[j].elapsed_time(evs[j + 1]) for j in range(len(names))])
        pt = torch.tensor(acc / (frames_p - 1), dtype=torch.float64, device="cuda")
        pmax = pt.clone(); dist.all_reduce(pmax, op=dist.ReduceOp.MAX); pmin = pt.clone(); dist.all_reduce(pmin, op=dist.ReduceOp.MIN)
        phases = {"ms_max_over_ranks": dict(zip(names, [float(x) for x in pmax])), "ms_min_over_ranks": dict(zip(names, [float(x) for x in pmin])),
                  "note": "CUDA events on the launching stream between the phases of one frame, mean of 5 frames, each frame followed by a synchronize (so `all_gather` includes waiting for the slowest rank's path_trace)"}

    # ---- end-to-end through the C ABI with host buffers: constants in, accumulated RGBA32F image out, every step -------------------------
    barrier()
    t0 = time.perf_counter()
    for i in range(args.steps):
        consts.sampleBaseIndex = (args.warmup + args.steps + i) * SPP
        if world == 1:
            ctx.render_frame(consts, 0, SPP, host_out)      # set_constants + path_trace + blocking read-back into host memory, on the context's own stream
        else:
            frame(args.warmup + args.steps + i)
            torch.cuda.synchronize()
            ctx.readback_accumulated(host_out)
    barrier()
    e2e_s = time.perf_counter() - t0
    e2e_t = torch.tensor([e2e_s], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(e2e_t, op=dist.ReduceOp.MAX)
    e2e_value = rays_per_frame / (float(e2e_t[0]) / args.steps) / 1e6

    # ---- roofline of the dominant kernel (closest-hit traversal): instrumented frame for N_node / N_tri, then algorithmic bytes / time ------
    roofline = None; launches = st.kernelLaunches; paths = st.paths
    rays_per_bounce = [int(x) for x in st.raysPerBounce[:BOUNCES + 2]]
    scatter, shadow = int(st.scatterRays), int(st.shadowRays)
    if rank == 0:
        ctx2 = lib.Context(max_sub_samples_per_launch=SPP, device=local_rank, tile_rank=rank if not emulate else 0, tile_world=world if not emulate else emulate, tile_size=64, flags=S.CFG_COUNT_TRAVERSAL_STEPS)
        ctx2.upload_scene(scene); consts.sampleBaseIndex = (args.warmup + args.steps - 1) * SPP; ctx2.set_constants(consts)
        ctx2.path_trace(0, SPP, True); ctx2.synchronize(); s2 = ctx2.stats(); ctx2.close()
        # per-kernel times: a context with CUDA events around every launch (RTXPT_CFG_TIME_KERNELS runs the kernels back to back, without the
        # shadow/closest overlap of the measured configuration), same frames, 3 warm-up + 1 measured
        ctx3 = lib.Context(max_sub_samples_per_launch=SPP, device=local_rank, tile_rank=rank if not emulate else 0, tile_world=world if not emulate else emulate, tile_size=64, flags=S.CFG_TIME_KERNELS)
        ctx3.upload_scene(scene)
        for i in range(4):
            consts.sampleBaseIndex = (args.warmup + args.steps - 4 + i) * SPP; ctx3.set_constants(consts); ctx3.path_trace(0, SPP, True)
        ctx3.synchronize(); s3 = ctx3.stats(); ctx3.close()
        k_closest, k_shadow, k_shade, k_other = s3.msTraceClosest, s3.msTraceShadow, s3.msShade, s3.msOther
        alg_bytes = 48 * s2.scatterRays + 80 * s2.traversalNodeVisits + 48 * s2.traversalTriTests      # SURVEY.md §8d: 32 B ray in + 16 B hit out + 80 B/node + 48 B/triangle
        peak, peak_src = measured_peak_gbs()
        achieved = alg_bytes / (k_closest * 1e-3) / 1e9 if k_closest > 0 else 0.0
        cap = ncu_capture(rays_per_bounce)
        dram_gbs = (cap["capture_dram_bytes"] / (cap["capture_ms"] * 1e-3) / 1e9) if cap.get("capture_ms") else None
        # The traversal kernel is bound by instruction issue, not by HBM (profiles/): `frac` stays the contract's algorithmic-bytes figure (SURVEY §8d: what the kernel would
        # have to move if nothing were cached, over its time and the measured HBM peak); `frac_dram` is what ncu saw cross the DRAM interface, `issue_active` the share of
        # issue slots in use - the number the kernel is actually limited by - and `thread_inst_per_ray` the quantity to drive down.
        roofline = {"kernel": "k_trace_closest (CWBVH8 closest-hit traversal)", "bound": "issue", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                    "frac_basis": "algorithmic bytes (48 B/ray + 80 B/node visit + 48 B/triangle test) / kernel time / measured HBM peak",
                    "traffic": cap.get("traffic"), "traffic_note": cap.get("note"), "traffic_capture_commit": cap.get("commit"),
                    "frac_dram": (dram_gbs / peak) if dram_gbs else None, "dram_gbs": dram_gbs,
                    "issue_active": cap.get("issue_active"), "threads_per_inst": cap.get("threads_per_inst"), "thread_inst_per_ray": cap.get("thread_inst_per_ray"),
                    "peak_source": peak_src,
                    "algorithmic_bytes_per_frame": int(alg_bytes), "nodes_per_ray": s2.traversalNodeVisits / max(1, s2.scatterRays), "tris_per_ray": s2.traversalTriTests / max(1, s2.scatterRays),
                    "kernel_ms_per_frame": {"trace_closest": k_closest, "trace_shadow": k_shadow, "shade": k_shade, "other": k_other},
                    "note": "kernel times: CUDA events around every launch of one frame in a separate RTXPT_CFG_TIME_KERNELS context (kernels serialised, one pipeline lane; the measured configuration overlaps k_trace_shadow(i) with k_trace_closest(i+1) and runs the frame's sub-samples as pipeline lanes)"}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        r = run_cpu(scene, consts, 3, 1)
        cpu = {"value": r["mrays_s"], "unit": "Mrays/s", "cores": r["threads"], "kind": "port", "sample": r["sample"], "bvh_build_s": r["bvh_build_s"], "rays_per_path": r["rays_per_path"],
               "cores_busy": r["cores_busy"], "host_cpus": r["host_cpus"], "loadavg": r["loadavg"]}

    realtime = None
    if rank == 0 and world == 1 and not args.no_realtime:
        # realtime mode (row a17) timed in a child process on the same workload: a fault there cannot take the headline line with it
        try:
            r = subprocess.run([sys.executable, "-B", os.path.join(os.path.dirname(os.path.abspath(__file__)), "scripts", "bench_realtime.py")], capture_output=True, text=True, timeout=300)
            # the child prints its line before tearing the context down, so a fault in its last (never-before-run) stage still leaves the measurements
            realtime = json.loads(r.stdout.strip().splitlines()[-1]) if r.stdout.strip() else {"error": "exit %d: %s" % (r.returncode, r.stderr.strip()[-300:])}
            if r.returncode != 0: realtime["child_exit"] = r.returncode
        except Exception as e:        # timeout, malformed output
            realtime = {"error": repr(e)[:300]}

    if rank == 0:
        line = {"metric": "Mrays/s", "value": value, "unit": "Mrays/s", "n_gpus": n_gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step,
                "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32 (fp16 path-state storage)", "data": "synthetic",
                "config": workload_config(n_gpus),
                "e2e": {"value": e2e_value, "unit": "Mrays/s", "h2d_bytes_per_step": C.sizeof(type(consts)), "d2h_bytes_per_step": WIDTH * HEIGHT * 16,
                        "ms_per_step": float(e2e_t[0]) / args.steps * 1e3},
                "gpu_launches": int(launches * args.steps),
                "rays_per_frame": rays_per_frame, "rays_per_path": rays_per_frame / (WIDTH * HEIGHT * SPP), "scatter_rays": scatter, "shadow_rays": shadow,
                "rays_per_iteration": rays_per_bounce, "bvh_build_s": st.bvhBuildSeconds, "bvh_nodes": st.bvhNodeCount, "lights": st.lightCount,
                "emulated_world": emulate or None, "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu, "phases": phases,
                "config3": (realtime or {}).get("config3") if isinstance(realtime, dict) else None, "realtime": realtime}
        sys.stdout.flush(); os.write(real_stdout, (json.dumps(line) + "\n").encode())
    ctx.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
