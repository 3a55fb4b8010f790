#!/usr/bin/env python
"""bench.py -- B-SHOT front-end benchmark (contract: see the task prompt / DESIGN.md section 6).

  python bench.py [--gpus N] [--steps K] [--warmup W]            # this repo's CUDA path
  python bench.py --impl reference [--gpus N] ...               # CPU oracle port, host cores, same config
  torchrun ... bench.py --gpus N ...                            # one rank per GPU (N > 1)
  python bench.py ... --dump-outputs DIR                        # + the last timed frame's outputs as DIR/<name>.npy

Headline workload (config.workload = "C3", BASELINE.json configs[2], the north_star frame and the largest
single-GPU configuration): HDL-64E-shaped 120 000-ray scans, 10 000 keypoints per frame, frame-to-frame:
voxel build -> seg-ratio detector -> top-K -> normals -> SHOT LRF + 352-bin histogram -> B-SHOT bits -> Hamming
mutual-NN match against the previous frame.  One step = one frame.  metric = B-SHOT descriptors/s through that
whole path.  The detector / normals run in the only mode there is: the reference's fp32 summation order
(bit-identical scores and keypoint indices, tests/test_detector_edge_gpu.py).
 * value : cloud already resident in HBM when the timed region starts (bshot_process_frame_dev).
 * e2e   : the C-ABI call a reference maintainer would make (bshot_process_frame) on pinned HOST buffers,
           H2D + D2H inside the timed region.
 * N > 1 : frame extraction does not shard (SURVEY 8e: replicas only) -> every rank processes a replica of the
           frame stream, no data-path collective, weak scaling.  The part of the path that DOES shard -- frame-to-
           map Hamming search against a map split over the ranks -- is timed in the same run and reported under
           "map_match" (C4: Q = 10 000 / 2 048 / 600 queries vs T = 1 048 576 map descriptors, with the single-GPU
           time of the same search measured in the same run -> efficiency_vs_1gpu; C5: T = 16 777 216 when 8 ranks)
           for the north_star's XOR + POPC kernel, and under "map_match_tc" for the tensor-core pipeline (tcgen05
           kind::i8, hamming_tc2.cu) that the library picks by itself for searches of this size -- same bit-exact result.
 * extra objects at N = 1: "c2" (BASELINE.json configs[1]: HDL-32E sequence, K = 2 048, per-frame p50 / p99 over
           500 distinct frames), "c3_radius_sweep" (extraction throughput over the SHOT radius, FULL normals).
 * --impl reference: the oracle port of the reference's CPU path on all host cores, same config / frames / metric.
 * --dump-outputs DIR: what the last timed step of the headline path computed, as a caller of bshot_process_frame_dev
           receives it (bshot_fetch_frame), in float arrays so that two builds can be compared output for output: kp_idx
           (K), descriptor_bits (K x 352, one 0 / 1 per bit) and pairs (P x 2, query / target keypoint ordinals).  The
           frames are seeded, so the same arguments give the same inputs on every run.
The benchmark writes nothing into the source tree (no bytecode either): that tree may be read-only.
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True
sys.path.insert(0, os.path.join(ROOT, "tests"))
from conftest import load_bshot, load_oracle, load_sharded, load_synth  # noqa: E402  (loaders only, no pytest needed)

HBM_FALLBACK_GBS = 6650.0   # /opt/skills/guides/B200_PROFILING.md fallback
L2_FLUSH_BYTES = 256 << 20
WORKLOADS = {  # name: (sensor, rays per frame, keypoints per frame, distinct frames cycled)
    "C3": ("hdl64e", 120000, 10000, 8),
    "C2": ("hdl32e", 69440, 2048, 12),
}
METRIC, UNIT = "bshot_frontend_descriptors_per_s", "descriptors/s"
DUMP_LIMIT_BYTES = 64 << 20


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return HBM_FALLBACK_GBS, "fallback (B200_PROFILING.md)"


def int8_peak_tops():
    """dense int8 tensor peak in TOP/s: twice the measured cuBLAS bf16 burst figure (int8 is nominally 2 x bf16 on B200; the
    pool has no measured int8 GEMM), else twice the profiling guide's fallback"""
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return 2.0 * float(json.load(open(p))["bf16_tflops"]), "2 x measured bf16 burst (MEASURED_PEAKS.json)"
    except Exception:
        return 2.0 * 1590.0, "2 x fallback bf16 (B200_PROFILING.md)"


class ClockSampler:
    """SM clock / throttle reasons sampled in-process through NVML every ~2 ms while `active` (the timed regions last
    tens of milliseconds: an external nvidia-smi loop at 100 ms sees nothing)."""

    def __init__(self, gpu_index):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self.active, self.stop_flag, self.thread, self.nv = False, False, None, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.thread = threading.Thread(target=self._run, daemon=True)
            self.thread.start()
        except Exception:
            self.nv = None

    def _run(self):
        nv = self.nv
        names = {"hw_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4)}
        while not self.stop_flag:
            if self.active:
                try:
                    self.samples.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                    for k, bit in names.items():
                        if r & bit:
                            self.reasons.add(k)
                except Exception:
                    pass
            time.sleep(0.002)

    def stop(self):
        self.stop_flag = True
        if self.thread:
            self.thread.join(timeout=1.0)
        out = {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples),
               "how": "NVML in-process, ~2 ms period, during the timed regions (value + e2e)"}
        if self.samples:
            out["sm_mhz"] = float(np.median(self.samples))
        return out


def workload_config(name, top_k, normals, points_per_frame):
    """the workload-defining keys -- identical in the CUDA arm and in the --impl reference arm"""
    sensor, rays, _, nframes = WORKLOADS[name]
    return {"workload": name, "sensor": sensor, "rays_per_frame": rays, "points_per_frame": int(points_per_frame), "top_k": int(top_k),
            "radius_mm": 3000, "max_nn": 300, "sr_type": "CV", "normals": normals.upper(), "frames_cycled": nframes,
            "match": "frame-to-frame mutual nearest neighbour (initial frame against itself)"}


def make_frames(synth, name):
    sensor, _, _, nframes = WORKLOADS[name]
    return [synth.make_scan(sensor, f) for f in range(nframes)]


def cpu_front_end(oracle, scans, top_k, threads, detector_threads=None, prev=None):
    """the oracle port of the reference path on host cores; returns (seconds per frame, last descriptors)"""
    t0 = time.perf_counter()
    for xyz in scans:
        c = oracle.Cloud(xyz)
        ratio = c.seg_ratio(3000.0, 300, oracle.SR_CV, threads=detector_threads or threads)
        idx, _ = oracle.select_keypoints(ratio, top_k, oracle.TIE_STDSORT)
        d = c.compute_descriptors(xyz[idx], 3000.0, 300, oracle.MODE_REFERENCE, threads=threads)
        tgt = d["bits"] if prev is None else prev
        m = oracle.match(d["bits"], tgt, want_right=True, threads=detector_threads or threads)
        oracle.mutual(m["left_idx"], m["right_idx"])
        prev = d["bits"]
    return (time.perf_counter() - t0) / len(scans), prev


def run_reference(args, rank):
    """--impl reference: the reference's CPU path (oracle port; only include/bshot_bits.h of the reference compiles
    here, DESIGN.md section 5) on all host cores: same workload, frames, metric and steps as the CUDA arm; every step
    is one whole frame (about a second on 16 cores)."""
    if rank != 0:
        return
    oracle, synth = load_oracle(), load_synth()
    cores = os.cpu_count() or 1
    frames = make_frames(synth, args.workload)
    W, K = max(args.warmup, 3), args.steps
    prev = None
    for i in range(W):
        _, prev = cpu_front_end(oracle, [frames[i % len(frames)]], args.top_k, cores, prev=prev)
    per = []
    for s in range(K):
        t, prev = cpu_front_end(oracle, [frames[(W + s) % len(frames)]], args.top_k, cores, prev=prev)
        per.append(t)
    sec = float(np.mean(per))
    val = args.top_k / sec
    sample = f"{K} whole frames of this workload (detector + top-K + normals + SHOT + B-SHOT + match), OpenMP over {cores} threads"
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": K, "warmup": W,
        "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32/f64+u32",
        "data": "synthetic", "config": workload_config(args.workload, args.top_k, args.normals, np.mean([len(f) for f in frames])),
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def dump_outputs(out_dir, synth, frame):
    """one frame's outputs (Context.fetch_frame) as DIR/<name>.npy in float32 / float64; above DUMP_LIMIT_BYTES in all,
    descriptor_bits keeps a seeded sample of its rows and descriptor_rows says which"""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"kp_idx": frame["kp_idx"].astype(np.float64), "pairs": frame["pairs"].astype(np.float64)}
    bits = synth.unpack_bits(frame["bits"]).astype(np.float32)
    room = DUMP_LIMIT_BYTES - sum(a.nbytes for a in arrays.values())
    if bits.nbytes > room:
        rows = np.sort(np.random.default_rng(0).choice(len(bits), room // (bits.shape[1] * 4 + 8), replace=False))
        arrays["descriptor_rows"] = rows.astype(np.float64)
        bits = bits[rows]
    arrays["descriptor_bits"] = bits
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def percentile_summary(x):
    x = np.asarray(x, dtype=np.float64)
    return {"mean": float(x.mean()), "p50": float(np.percentile(x, 50)), "p90": float(np.percentile(x, 90)),
            "p99": float(np.percentile(x, 99)), "max": float(x.max()), "frames": int(len(x))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="C3", choices=sorted(WORKLOADS))
    ap.add_argument("--top-k", dest="top_k", type=int, default=None)
    ap.add_argument("--normals", default="reference", choices=["reference", "full"])
    ap.add_argument("--map-t", type=int, default=1 << 20)
    ap.add_argument("--map-steps", type=int, default=10)
    ap.add_argument("--no-map", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the C2 sequence and the C3 SHOT-radius sweep objects")
    ap.add_argument("--map-only", action="store_true", help="debug: print only the map_match object")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed frame's outputs to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.top_k is None:
        args.top_k = WORKLOADS[args.workload][2]

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs: the outputs are those of the CUDA path (--impl ours)")
        run_reference(args, rank)
        return

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    bs, synth = load_bshot(), load_synth()
    W = max(args.warmup, 3)
    K = args.steps
    hbm_peak, peak_src = peaks()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- inputs ---------------------------------------------------------------------------------
    # replicas: every rank runs the SAME frames (identical work per GPU keeps the weak-scaling figure clean)
    frames = make_frames(synth, args.workload)
    nfr = len(frames)
    npts = [len(f) for f in frames]
    max_n = max(npts)
    mode = bs.NORMALS_REFERENCE if args.normals == "reference" else bs.NORMALS_FULL
    params = bs.default_params(top_k=args.top_k, normals_mode=mode)
    map_q = 10000
    ctx = bs.Context(local_rank, max_points=max_n + 1024, max_keypoints=max(args.top_k, map_q),
                     max_targets=max(args.top_k, (args.map_t + world - 1) // world, args.map_t if world > 1 else 0,
                                     (1 << 24) // world if world == 8 else 0))
    st = torch.cuda.ExternalStream(ctx.stream)
    d_frames = [torch.from_numpy(f).cuda() for f in frames]                 # resident in HBM
    h_frames = [torch.from_numpy(f).pin_memory() for f in frames]           # pinned host copies
    h_kp = torch.empty(args.top_k, dtype=torch.int32).pin_memory()
    h_bits = torch.empty((args.top_k, 6), dtype=torch.int64).pin_memory()
    h_pairs = torch.empty((args.top_k, 2), dtype=torch.int32).pin_memory()
    flush = torch.empty(L2_FLUSH_BYTES // 4, dtype=torch.float32, device="cuda")

    def l2_flush():
        with torch.cuda.stream(st):
            flush.fill_(1.0)

    def step_resident(i):
        f = i % nfr
        ctx.process_frame_dev(d_frames[f].data_ptr(), npts[f], 12, params)

    def step_e2e(i):
        f = i % nfr
        return ctx.process_frame_raw(h_frames[f].data_ptr(), npts[f], 12, params, h_kp.data_ptr(),
                                     h_bits.data_ptr(), h_pairs.data_ptr())

    # ---- HBM-resident timing (value) ---------------------------------------------------------------
    sampler = ClockSampler(local_rank) if rank == 0 else None
    ctx.enable_timing(True)
    for i in range(W):
        step_resident(i)
    ctx.sync()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    stage_acc, counters_acc = {}, {}
    launches0 = ctx.launch_count()
    barrier()
    if sampler:
        sampler.active = True
    for i in range(K):
        l2_flush()
        ev[i][0].record(st)
        step_resident(W + i)
        ev[i][1].record(st)
        for k, v in ctx.stage_times().items():      # synchronises; outside the event pair
            stage_acc[k] = stage_acc.get(k, 0.0) + v
        for k, v in ctx.frame_counters().items():
            counters_acc[k] = counters_acc.get(k, 0) + v
    barrier()
    if sampler:
        sampler.active = False
    launches = ctx.launch_count() - launches0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, synth, ctx.fetch_frame(args.top_k))
    per_step = [a.elapsed_time(b) for a, b in ev]
    ms_total = max_over_ranks(sum(per_step))
    ms_step = ms_total / K
    n_desc = counters_acc["keypoints"] / K                       # descriptors actually produced per frame
    value = world * n_desc / (ms_step * 1e-3)
    stages = {k: v / K for k, v in stage_acc.items()}

    # ---- roofline of the dominant kernel (and the others beside it) ---------------------------------------
    # algorithmic bytes per launch (SURVEY 8d): 16 B per selected neighbour (+ 16 B per neighbour normal in SHOT) + outputs
    mean_n = float(np.mean(npts))
    kern = {"seg_ratio": ("tile_kernel + tile_single_kernel (seg-ratio detector stage)", 16.0 * counters_acc["detector_neighbours"] / K + 12.0 * mean_n),
            "shot_bshot": ("shot_kernel", 32.0 * counters_acc["shot_neighbours"] / K + 48.0 * n_desc),
            # REFERENCE normals of the frame path: the neighbour reads happened in the detector pass (covariance sums kept per point);
            # what is left is 40 B of sums in + 16 B out per keypoint
            "normals": ("normals_from_sums_kernel (sums kept by the detector pass)", 56.0 * n_desc),
            "voxel_build": ("grid_build", 2 * 16.0 * mean_n)}
    traffic_tab = {}
    try:
        traffic_tab = json.load(open(os.path.join(ROOT, "profiles", "traffic_r3.json")))
    except Exception:
        pass

    def roof(name):
        kname, alg = kern[name]
        ach = alg / (stages[name] * 1e-3) / 1e9
        t = traffic_tab.get(name, {})
        r = {"bound": "hbm", "kernel": kname, "achieved": ach, "peak": hbm_peak, "unit": "GB/s", "frac": ach / hbm_peak,
             "traffic": t.get("dram_bytes_per_launch"), "peak_source": peak_src, "algorithmic_bytes_per_launch": alg,
             "ms_per_launch": stages[name], "ncu": t.get("ncu")}
        if t.get("warp_instructions_per_launch") and args.workload == "C3":
            # what actually bounds the kernel: warp instructions (counted by ncu on this workload) against the issue slots
            # of the launch's live duration (4 schedulers per SM, one instruction per clock)
            sm_clock = (clock_probe or {}).get("sm_max_mhz") or 1965.0
            peak_issue = torch.cuda.get_device_properties(local_rank).multi_processor_count * 4 * sm_clock * 1e6
            wi = float(t["warp_instructions_per_launch"])
            r["issue"] = {"warp_instructions_per_launch": wi, "achieved_warp_inst_per_s": wi / (stages[name] * 1e-3),
                          "peak_warp_inst_per_s": peak_issue, "frac": wi / (stages[name] * 1e-3) / peak_issue,
                          "source": "instruction count: ncu smsp__inst_executed.sum (profiles/r3z_ncu_full.txt); time: this run"}
        return r
    clock_probe = {"sm_max_mhz": sampler.max_mhz} if sampler and sampler.max_mhz else None
    dom = max(kern, key=lambda k: stages[k])
    roofline = roof(dom)
    roofline["note"] = ("the cloud (< 2 MB) is L2 resident and the neighbourhood tiles are staged once per block in shared memory: "
                        "the algorithmic bytes are re-read from shared memory, not HBM; the kernel is bound by instruction issue "
                        "(DESIGN.md section 7)")
    roofline_others = {k: roof(k) for k in kern if k != dom}

    # ---- end-to-end through the host-buffer C ABI (e2e) ---------------------------------------------
    ctx.enable_timing(False)
    for i in range(W):
        step_e2e(i)
    barrier()
    if sampler:
        sampler.active = True
    t_e2e = 0.0
    for i in range(K):
        l2_flush()
        ctx.sync()
        t0 = time.perf_counter()
        step_e2e(W + i)
        t_e2e += time.perf_counter() - t0
    barrier()
    clocks = sampler.stop() if sampler else None
    t_e2e = max_over_ranks(t_e2e)
    e2e_val = world * n_desc / (t_e2e / K)
    e2e = {"value": e2e_val, "unit": UNIT, "ms_per_step": t_e2e / K * 1e3,
           "h2d_bytes_per_step": int(mean_n * 12),
           "d2h_bytes_per_step": int(args.top_k * (4 + 48 + 12) + 8),
           "api": "bshot_process_frame (C ABI, pinned host buffers, synchronous)"}

    # ---- sharded frame-to-map matching (the part of the path that shards) -----------------------------
    map_match = map_match_tc = None
    if not args.no_map:
        map_match = bench_map(args, bs, synth, ctx, st, world, rank, local_rank, barrier, max_over_ranks, kind=0)
        map_match_tc = bench_map(args, bs, synth, ctx, st, world, rank, local_rank, barrier, max_over_ranks, kind=2)
        ctx.set_matcher(-1)

    # ---- extras at N = 1 ------------------------------------------------------------------------------
    c2 = c3_sweep = pose_loop = None
    if rank == 0 and world == 1 and not args.no_extras and not args.map_only:
        def extra(fn, *a):   # an extra object never takes the headline line down with it
            try:
                return fn(*a)
            except Exception as e:
                return {"error": f"{type(e).__name__}: {e}"}
        c2 = extra(bench_c2_sequence, bs, synth, local_rank, flush)
        c3_sweep = extra(bench_c3_sweep, bs, synth, local_rank, flush)
        pose_loop = extra(bench_pose_loop, bs, synth, local_rank)

    # ---- CPU baseline (rank 0, N = 1 only; bounded sample) --------------------------------------------
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu and not args.map_only:
        oracle = load_oracle()
        cores = os.cpu_count() or 1
        cpu_front_end(oracle, frames[:1], args.top_k, cores)      # warm-up (page-in, OpenMP pool)
        sample = frames[:min(nfr, 6)]
        sec, _ = cpu_front_end(oracle, sample, args.top_k, cores)
        sec_ref, _ = cpu_front_end(oracle, sample[:1], args.top_k, min(12, cores), detector_threads=1)
        cpu_baseline = {"value": args.top_k / sec, "unit": UNIT, "cores": cores, "kind": "port", "ms_per_frame": sec * 1e3,
                        "sample": f"{len(sample)} whole frames of this workload (detector + top-K + normals + SHOT + B-SHOT + match), all cores",
                        "reference_threading": {"value": args.top_k / sec_ref, "ms_per_frame": sec_ref * 1e3, "detector_match_threads": 1,
                                                "normals_shot_threads": min(12, cores), "sample": "1 frame"}}

    if rank == 0 and args.map_only:
        print(json.dumps({"map_match": map_match, "map_match_tc": map_match_tc}))
    elif rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32/f64+u32", "data": "synthetic",
            "config": workload_config(args.workload, args.top_k, args.normals, mean_n),
            "timing": {"l2": f"flushed between steps ({L2_FLUSH_BYTES >> 20} MiB write)", "clock": "per-step CUDA events on the context stream",
                       "parallelism": "replicas (one frame stream per GPU, no data-path collective)" if world > 1 else "single GPU",
                       "ms_per_step_distribution": percentile_summary(per_step), "descriptors_per_frame": n_desc,
                       "detector_mode": "exact: fp32 running sums replayed in neighbour order (scores / keypoint indices bit-identical to the oracle)"},
            "stages_ms": stages, "roofline": roofline, "roofline_others": roofline_others, "cpu_baseline": cpu_baseline, "e2e": e2e,
            "gpu_launches": int(launches), "clocks": clocks, "map_match": map_match, "map_match_tc": map_match_tc, "c2": c2, "c3_radius_sweep": c3_sweep, "pose_loop": pose_loop,
        }
        print(json.dumps(line))
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


def bench_map(args, bs, synth, ctx, st, world, rank, local_rank, barrier, max_over_ranks, kind=0):
    """C4 / C5: Q queries vs a T-descriptor map split over the ranks; per-call device time (max over ranks), the single-GPU
    time of the SAME search in the same run (-> efficiency_vs_1gpu) and the roofline of the distance-matrix kernel:
    kind 0 = XOR + POPC (POPC pipe), kind 2 = tensor-core pipeline (int8 tensor peak)."""
    import torch
    sharded = load_sharded()
    dev = torch.device("cuda", local_rank)
    ctx.set_matcher(kind)
    popc_peak = ctx.popc_peak()
    i8_peak, i8_src = int8_peak_tops()
    rows = []

    def timed(fn, reps):
        fn(); fn()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = ctx.launch_count()
        e0.record(st)
        for _ in range(reps):
            fn()
        e1.record(st)
        barrier()
        return max_over_ranks(e0.elapsed_time(e1)) / reps, (ctx.launch_count() - l0) // reps

    def device_map(T, seed):
        """map descriptors generated on the device (i.i.d. 352-bit words; word 5 keeps only its low 32 bits)"""
        g = torch.Generator(device=dev)
        g.manual_seed(seed)
        m = torch.randint(-2 ** 63, 2 ** 63 - 1, (T, 6), dtype=torch.int64, device=dev, generator=g)
        m[:, 5] &= 0xFFFFFFFF
        return m

    configs = [("C4", args.map_t, q) for q in (10000, 2048, 600)]
    if world == 8:
        configs.append(("C5", 1 << 24, 10000))
    for name, T, Q in configs:
        per = (T + world - 1) // world
        lo, hi = rank * per, min(T, (rank + 1) * per)
        if name == "C4":
            tfull = synth.random_descriptors(T, seed=7)            # same global map on every rank
            q = synth.random_descriptors(Q, seed=8)
            planted = np.random.default_rng(9).permutation(T)[:64]  # self-check: 64 queries are exact copies of map entries
            q[:64] = tfull[planted]
            dq = torch.from_numpy(q.view(np.int64)).to(dev)
            # single-GPU time of the same search, measured in this run (world > 1 only; at world 1 it IS the measurement)
            t1 = None
            if world > 1:
                ctx.map_reset()
                ctx.map_append(tfull)
                single = sharded.DeviceShardedMatcher(ctx, 1, 0, Q, device=dev)
                t1, _ = timed(lambda: single.match(dq.data_ptr(), 0), max(3, args.map_steps // 2))
            ctx.map_reset()
            ctx.map_append(tfull[lo:hi])
            del tfull
        else:
            full = device_map(per, 1000 + rank)                     # C5: every rank generates its own shard on the device
            ctx.map_reset()
            ctx.map_append_dev(full.data_ptr(), per)
            hi = lo + per
            q = synth.random_descriptors(Q, seed=8)
            dq = torch.from_numpy(q.view(np.int64)).to(dev)
            planted, t1 = None, None
            del full
        matcher = sharded.DeviceShardedMatcher(ctx, world, rank, Q, mode=os.environ.get("BSHOT_EXCHANGE", "auto"), device=dev)
        last = matcher.match(dq.data_ptr(), lo)
        barrier()
        if planted is not None:
            rec = last[:64].cpu().numpy().view(bs.CAND_DTYPE).reshape(64)
            chk = bs.unpack_cands(rec)
            if not (np.array_equal(chk["idx1"], planted) and (chk["dist1"] == 0).all() and np.array_equal(chk["rq"], np.arange(64))):
                raise SystemExit("bench.py: sharded map match self-check failed (planted duplicates not recovered)")
        mm_ms, per_call = timed(lambda: matcher.match(dq.data_ptr(), lo), args.map_steps)
        matcher.check()
        pairs = float(Q) * float(T)
        if kind == 0:
            roof = {"bound": "popc", "achieved": 11 * pairs / (mm_ms * 1e-3) / 1e12, "peak": world * popc_peak / 1e12,
                    "unit": "TPOPC32/s", "frac": 11 * pairs / (mm_ms * 1e-3) / (world * popc_peak),
                    "issued_popc_per_pair": 6, "frac_of_issued": 6 * pairs / (mm_ms * 1e-3) / (world * popc_peak),
                    "peak_source": "measured live (bshot_popc_peak microbenchmark) x shards"}
        else:   # 352 multiply-adds per pair are the algorithm; the kernel issues 384 (one extra K step carries |q|, |t| and the column)
            roof = {"bound": "tensor", "achieved": 2 * 352 * pairs / (mm_ms * 1e-3) / 1e12, "peak": world * i8_peak, "unit": "TOP/s (int8)",
                    "frac": 2 * 352 * pairs / (mm_ms * 1e-3) / 1e12 / (world * i8_peak), "issued_k_per_pair": 384,
                    "frac_of_issued": 2 * 384 * pairs / (mm_ms * 1e-3) / 1e12 / (world * i8_peak), "peak_source": i8_src + " x shards"}
        row = {"workload": name, "Q": Q, "T": T, "shards": world, "kernel": "hamming_top2_kernel (XOR + POPC)" if kind == 0 else "hamming_tc2_kernel (tcgen05 kind::i8)",
               "ms_per_call": mm_ms, "pairs_per_s": pairs / (mm_ms * 1e-3),
               "target_GBps": T * 48 / (mm_ms * 1e-3) / 1e9, "roofline": roof,
               "collective": matcher.describe(), "gpu_launches_per_call": per_call}
        if world == 1:
            row["ms_per_call_1gpu"], row["efficiency_vs_1gpu"] = mm_ms, 1.0
        elif t1 is not None:
            row["ms_per_call_1gpu"], row["efficiency_vs_1gpu"] = t1, t1 / (world * mm_ms)
        rows.append(row)
        del matcher
    out = dict(rows[0])
    out["others"] = rows[1:]
    return out


def _scan_worker(job):
    sensor, f, pos, yaw = job
    return load_synth().make_scan(sensor, f, pos=pos, yaw_deg=yaw)


def loop_pose(k, n):
    """closed loop through the synthetic scene: out to x = 75 m and back with a 3 m sideways swing, <= 471 mm per frame at
    n = 500 (the reference drives ~500 mm per HDL-32E rotation), yaw 0.5 deg per frame"""
    a = 2.0 * np.pi * k / n
    return (37500.0 * (1.0 - np.cos(a)), 3000.0 * np.sin(a), 0.0), 0.5 * k


def make_sequence(sensor, n_frames):
    """n_frames distinct synthetic scans along loop_pose; the numpy ray caster runs on a pool of host processes (spawned:
    the parent already holds a CUDA context)"""
    import multiprocessing as mp
    from concurrent.futures import ProcessPoolExecutor
    workers = max(1, min(16, os.cpu_count() or 1))
    jobs = [(sensor, f) + loop_pose(f, n_frames) for f in range(n_frames)]
    try:
        with ProcessPoolExecutor(max_workers=workers, mp_context=mp.get_context("spawn")) as ex:
            return list(ex.map(_scan_worker, jobs, chunksize=4))
    except Exception as e:   # no pool on this host: every fourth pose of the same loop, ray-cast in this process
        print(f"bench.py: scan pool unavailable ({type(e).__name__}: {e}); serial fallback", file=sys.stderr)
        return [_scan_worker(j) for j in jobs[::4]]


def bench_c2_sequence(bs, synth, device, flush, n_frames=500, top_k=2048):
    """C2 (BASELINE.json configs[1]): frame-to-frame odometry front end over a 500-frame synthetic HDL-32E sequence -- per-frame
    device times over 500 DISTINCT frames (a closed loop through the scene, <= 471 mm and 0.5 deg of yaw per frame), L2 flushed
    before every frame"""
    import torch
    frames = make_sequence("hdl32e", n_frames)
    ctx = bs.Context(device, max_points=max(len(f) for f in frames) + 1024, max_keypoints=top_k, max_targets=top_k)
    st = torch.cuda.ExternalStream(ctx.stream)
    p = bs.default_params(top_k=top_k)
    d = [torch.from_numpy(f).cuda() for f in frames]
    for i in range(3):
        ctx.process_frame_dev(d[i].data_ptr(), len(frames[i]), 12, p)
    ctx.reset()
    ctx.sync()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in frames]
    for i, f in enumerate(frames):
        with torch.cuda.stream(st):
            flush.fill_(1.0)
        ev[i][0].record(st)
        ctx.process_frame_dev(d[i].data_ptr(), len(f), 12, p)
        ev[i][1].record(st)
    ctx.sync()
    ms = [a.elapsed_time(b) for a, b in ev]
    ctx.enable_timing(True)
    acc = {}
    for i in range(8):
        ctx.process_frame_dev(d[i].data_ptr(), len(frames[i]), 12, p)
        for k, v in ctx.stage_times().items():
            acc[k] = acc.get(k, 0.0) + v / 8
    ctx.close()
    return {"workload": "C2", "sensor": "hdl32e", "top_k": top_k, "points_per_frame": int(np.mean([len(f) for f in frames])),
            "ms_per_frame": percentile_summary(ms), "descriptors_per_s": top_k / (float(np.mean(ms)) * 1e-3), "stages_ms": acc,
            "slowest_frame": {"index": int(np.argmax(ms)), "points": int(len(frames[int(np.argmax(ms))])), "ms": float(np.max(ms)),
                              "note": "per-frame events bracket the launches: a host-side hiccup of the launching thread shows up here"}}


def bench_pose_loop(bs, synth, device, n_frames=12, top_k=600):
    """the reference's whole per-frame loop (test/odometry_test.cpp:143-184) from raw laser returns to a pose, every stage
    through the C ABI with HOST buffers: Preprocessor::run + extractKeypoints + computeDescriptors (bshot_extract_scan),
    featureMatching against the device-resident map (bshot_match_frame_to_map + bshot_ransac), evaluateEstimation
    (gate + ICP), updateMap.  Reference defaults: HDL-32E, K = 600.  Wall clock per frame (synchronous calls)."""
    import time
    rot = [synth.make_lasers("hdl32e", f) for f in range(n_frames)]
    p = bs.default_params(top_k=top_k)
    ctx = bs.Context(device, max_points=131072, max_keypoints=1024, max_targets=1 << 16)
    ctx.gmap_create(1 << 16, 4096)
    stage = {k: [] for k in ("extract_scan", "match_to_map", "ransac", "gate_icp", "map_update", "frame")}
    pose_ref, poses = np.eye(4, dtype=np.float32), []
    for rep in range(2):                                  # first pass warms up (scratch growth, module load)
        ctx.reset(); ctx.gmap_reset()
        pose_ref, poses = np.eye(4, dtype=np.float32), []
        for k, L in enumerate(rot):
            t0 = time.perf_counter()
            f = ctx.extract_scan(L["azimuth"], L["vertical"], L["distance"], L["ring_deg"], p, want_cloud=False)
            t1 = time.perf_counter()
            if k == 0:
                pairs, tgt = ctx.match_mutual(f["bits"], f["bits"])[0], f["kp_xyz"]
            else:
                r = ctx.match_frame_to_map(pose_ref[:3, 3], 100000.0, pose_ref[:3], target_cap=1 << 16)
                pairs, tgt = r["pairs"], r["target_xyz"]
            t2 = time.perf_counter()
            rs = ctx.ransac(f["kp_xyz"], tgt, pairs)
            t3 = time.perf_counter()
            ev = ctx.evaluate_estimation(rs["transform"], pose_ref, len(rs["pairs"]), f["kp_xyz"], tgt, run_icp=True)
            t4 = time.perf_counter()
            ctx.gmap_update_from_frame(ev["T_best"][:3]); ctx.frame_commit(); ctx.sync()
            t5 = time.perf_counter()
            pose_ref = ev["T_best"]
            poses.append(pose_ref[:3, 3].tolist())
            if rep == 1 and k > 0:
                for name, a, b in (("extract_scan", t0, t1), ("match_to_map", t1, t2), ("ransac", t2, t3), ("gate_icp", t3, t4),
                                   ("map_update", t4, t5), ("frame", t0, t5)):
                    stage[name].append((b - a) * 1e3)
    n_map = ctx.gmap_size()[0]
    ctx.close()
    return {"workload": "lasers -> pose, HDL-32E rotations (69 440 returns), K = 600, frame-to-map", "frames": n_frames - 1,
            "ms_per_frame_wall": {k: float(np.median(v)) for k, v in stage.items()}, "map_keypoints": int(n_map),
            "last_position_mm": poses[-1], "truth_last_position_mm": [500.0 * (n_frames - 1), 0.0, 0.0],
            "note": "medians of synchronous host-buffer calls incl. Python/ctypes overhead; the sensor moves 500 mm per frame along x"}


def bench_c3_sweep(bs, synth, device, flush, top_k=10000):
    """C3 (BASELINE.json configs[2]): extraction throughput (normals + LRF + SHOT352 + B-SHOT) over the SHOT radius, FULL normals"""
    import torch
    frames = [synth.make_scan("hdl64e", f) for f in range(3)]
    d = [torch.from_numpy(f).cuda() for f in frames]
    ctx = bs.Context(device, max_points=max(len(f) for f in frames) + 1024, max_keypoints=top_k, max_targets=top_k)
    st = torch.cuda.ExternalStream(ctx.stream)
    ctx.enable_timing(True)
    sweep = []
    for R in (500.0, 1000.0, 2000.0, 3000.0, 4000.0):
        ctx.reset()
        p = bs.default_params(top_k=top_k, normals_mode=bs.NORMALS_FULL, normal_radius=R, shot_radius=R)
        for i in range(2):
            ctx.process_frame_dev(d[i % 3].data_ptr(), len(frames[i % 3]), 12, p)
        ctx.sync()
        acc, nbr, reps = {}, 0, 6
        for i in range(reps):
            with torch.cuda.stream(st):
                flush.fill_(1.0)
            ctx.process_frame_dev(d[i % 3].data_ptr(), len(frames[i % 3]), 12, p)
            for k, v in ctx.stage_times().items():
                acc[k] = acc.get(k, 0.0) + v / reps
            nbr += ctx.frame_counters()["shot_neighbours"] / reps
        ext_ms = acc["normals"] + acc["shot_bshot"]
        sweep.append({"radius_mm": R, "normals_ms": acc["normals"], "shot_bshot_ms": acc["shot_bshot"], "frame_ms": acc["frame"],
                      "descriptors_per_s": top_k / (ext_ms * 1e-3), "shot_neighbours_per_keypoint": nbr / top_k,
                      "shot_algorithmic_GBps": 32.0 * nbr / (acc["shot_bshot"] * 1e-3) / 1e9})
    ctx.close()
    return {"workload": "C3", "sensor": "hdl64e", "top_k": top_k, "normals": "FULL (normal radius = SHOT radius)", "sweep": sweep,
            "note": "stage times from CUDA events on the context stream, L2 flushed before every frame; the detector keeps R = 3000"}


if __name__ == "__main__":
    main()
