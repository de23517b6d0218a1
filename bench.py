#!/usr/bin/env python
"""bench.py — SOS front-end frame-pairs/s on B200 (BASELINE.json metric), with per-kernel roofline fractions and the
CPU reference path timed beside it.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c2|c1|tiny] [--batch B] [--dump-outputs DIR]
    python bench.py --impl reference ...          # the reference's CPU path (OpenCV + NumPy) on this box's host cores

A "step" is one pass of the hot path over one batch of B new synthetic frames = B frame pairs (frame i-1 -> frame i):
2 remaps, 12 stereo bucket matches, lifting + triangulation, 2 temporal matches and one RANSAC per pair.
One JSON line is printed by rank 0.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "sos_frame_pairs_per_s"
UNIT = "frame-pairs/s"


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


# ---------------------------------------------------------------------------------------------------------------------
# clocks
# ---------------------------------------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.FIELDS}",
                                          "--format=csv,noheader,nounits", "-lms", "50"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        for ln in self.lines:
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0])); mx.append(float(parts[1]))
            except ValueError:
                continue
            for n, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------------------------
# CPU path (oracle) on a bounded sample
# ---------------------------------------------------------------------------------------------------------------------
def host_workload(name: str, seed: int):
    """Rig, scene, LUT maps and masks built WITHOUT the GPU (NumPy), for the CPU arm."""
    from oracle import geometry
    from vo_single_camera_sos_b200 import synth, workload
    c = workload.CONFIGS[name]
    rig = synth.make_rig(c["width"], c["height"], c["pano_cols"], seed=seed)
    scene = synth.make_scene(int(c["feat"] * 2.0), seed=seed)
    p = rig.pano
    maps, masks = {}, {}
    for which in ("top", "bot"):
        lo, hi = rig.elev_top if which == "top" else rig.elev_bot
        g = dict(zip(synth.GUM_FIELDS, rig.gum_vector(which)))
        maps[which] = geometry.lut_build(g, p["rows"], p["cols"], p["cyl_height_max"], p["cyl_height_min"], lo, hi)
        masks[which] = rig.mask(which)
    hyp = np.random.default_rng(seed + 7).integers(0, 2 ** 32, (c["n_hyp"], 3), dtype=np.uint64).astype(np.uint32)
    return rig, scene, maps, masks, hyp, c


class CpuPath:
    """One frame pair per call through oracle.pipeline (OpenCV with all its threads + NumPy)."""

    def __init__(self, name: str, seed: int, n_frames: int, score_mode: str, refine: str = "arun", moving: float = 0.0):
        import cv2
        from vo_single_camera_sos_b200 import synth
        self.rig, self.scene, self.maps, self.masks, self.hyp, self.c = host_workload(name, seed)
        self.mode = score_mode
        self.refine = refine
        self.thr = 1.0 - math.cos(math.radians(5.0)) if score_mode == "bearing" else 0.05
        self.traj = synth.make_trajectory(n_frames, seed=seed)
        self.threads = cv2.getNumThreads()
        self.pano_g = dict(self.rig.pano)
        base = synth.render_omni(self.rig, self.scene, self.traj[0])
        rng = np.random.default_rng(seed)
        self.frames = []
        for i in range(n_frames):
            f = synth.make_frame_features(self.rig, self.scene, self.traj[i], self.c["feat"], 12, seed=1000 * i + 17,
                                          cap=self.c["cap"], dynamic=moving)
            # one rendered view of the scene + a per-frame noise variant (content does not change the work done)
            omni = base if i == 0 else np.bitwise_xor(base, rng.integers(0, 8, base.shape, dtype=np.uint8))
            self.frames.append((omni, f))
        self.rigm = np.zeros((2, 3, 4)); self.rigm[:, :, :3] = np.eye(3)
        self.rigm[0, :, 3] = self.rig.f_top; self.rigm[1, :, 3] = self.rig.f_bot
        self.state = None
        self.cursor = 0
        self.timer = {}           # seconds per stage, accumulated over pair() calls
        self.hyp_limit = None     # score only the first hyp_limit hypotheses (the reference's own budget is 210)
        self.bg_state = {}

    def _frame(self, i):
        from oracle import pipeline
        omni, f = self.frames[i % len(self.frames)]
        panos = pipeline.remap_views(omni, self.maps, self.masks, background_state=self.bg_state, timer=self.timer)
        n_t, n_b = f["top"]["bucket_off"][-1], f["bot"]["bucket_off"][-1]
        st = pipeline.stereo_frame(self.pano_g, self.rig.f_top, self.rig.f_bot, f["top"]["px"][:n_t], f["top"]["desc"][:n_t],
                                   f["top"]["bucket_off"], f["bot"]["px"][:n_b], f["bot"]["desc"][:n_b],
                                   f["bot"]["bucket_off"], cap=self.c["cap"], timer=self.timer)
        st["panos"] = panos
        return st

    def prime(self):
        self.state = self._frame(0)
        self.cursor = 1

    def pair(self):
        from oracle import pipeline
        cur = self._frame(self.cursor)
        out = pipeline.track_pair(self.state, cur, self.hyp, self.mode, self.thr, self.rigm,
                                  0.125 * 0.5 * self.rig.pano["cols"], refine=self.refine, hyp_limit=self.hyp_limit,
                                  timer=self.timer)
        self.state = cur
        self.cursor += 1
        return out


REF_BUDGET_S = 150.0   # wall-clock bound of the reference arm's timed region


def run_reference_c4(args):
    """CPU arm of config 4: the NumPy float64 RANSAC restatement (oracle/ransac.py; OpenGV absent) on the same 50 000
    correspondences and a bounded slice of the 65 536 hypotheses; the rate is per (hypothesis, correspondence) pair."""
    from oracle import ransac
    p_ref, p_cur, hyp = c4_problem()
    n = p_ref.shape[1]
    ransac.ransac_p3d(p_ref[0], p_cur[0], hyp[:4], "euclid", 0.05)   # warm-up
    t0 = time.perf_counter()
    done = 0
    chunk = 64
    while done < hyp.shape[0]:
        ransac.ransac_p3d(p_ref[0], p_cur[0], hyp[done:done + chunk], "euclid", 0.05)
        done += chunk
        if time.perf_counter() - t0 > 20.0:
            break
    dt = time.perf_counter() - t0
    value = float(n) * done / dt
    line = {"impl": "reference", "metric": "ransac_hypothesis_point_pairs_per_s", "value": value, "unit": "pairs/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / done * hyp.shape[0] * 1e3,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"c4: {n} 3D-3D correspondences x {hyp.shape[0]} hypotheses, euclid score, 35 % inliers",
                       "note": f"bounded sample: the first {done} hypotheses; ms_per_step extrapolates linearly to all of them"},
            "cpu_baseline": {"value": value, "unit": "pairs/s", "cores": 1, "kind": "port",
                             "sample": f"{done} of {hyp.shape[0]} hypotheses x {n} correspondences, NumPy float64 (single thread)"},
            "e2e": {"value": value, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def run_reference(args, rank, world):
    if rank != 0:
        return
    if args.workload == "c4":
        return run_reference_c4(args)
    seq = args.workload == "c3"          # config 3 runs the c1 geometry; its unit is the frame (one pair per new frame)
    if seq:
        args.workload = "c1"
    t_build = time.perf_counter()
    cpu = CpuPath(args.workload, seed=0, n_frames=min(args.steps + args.warmup + 1, 6), score_mode=args.score, refine=args.refine,
                  moving=args.moving)
    cpu.prime()
    # a C2 frame pair costs the CPU path seconds: the whole run is bounded to about REF_BUDGET_S by timing at most as many
    # steps as fit (the rate is what the line reports); warm-up pairs count against the budget too
    t_w = time.perf_counter()
    n_warm = 0
    for _ in range(args.warmup):
        cpu.pair()
        n_warm += 1
        if time.perf_counter() - t_w > REF_BUDGET_S / 4:
            break
    per_pair = (time.perf_counter() - t_w) / max(n_warm, 1) if n_warm else None
    t0 = time.perf_counter()
    inl = []
    timed = 0
    for _ in range(args.steps):
        o = cpu.pair()
        inl.append(o["best_count"] if o else -1)
        timed += 1
        el = time.perf_counter() - t0
        if el + (per_pair or el / timed) > REF_BUDGET_S:
            break
    dt = time.perf_counter() - t0
    value = timed / dt
    c = cpu.c
    line = {
        "impl": "reference", "metric": "sos_sequence_frames_per_s" if seq else METRIC, "value": value,
        "unit": "frames/s" if seq else UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / timed * 1e3, "higher_is_better": True, "scaling": "weak",
        "steps_timed": timed, "warmup_done": n_warm,
        "vs_baseline": None, "dtype": "u8/f64", "data": "synthetic",
        "config": workload_config(args, c, batch=1, note="reference arm: one frame pair per step (bounded sample)"),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cpu.threads, "kind": "port",
                         "sample": f"{timed} frame pairs of {args.workload} (of {args.steps} requested; the run is bounded to "
                                   f"{REF_BUDGET_S:.0f} s of CPU time); OpenCV calls as the reference makes them "
                                   f"({cpu.threads} threads) + NumPy float64; RANSAC = NumPy restatement (OpenGV absent)"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "setup_s": t0 - t_build, "ransac_inliers": inl,
    }
    print(json.dumps(line), flush=True)


def workload_config(args, c, batch, note=""):
    return {"workload": f"{args.workload}: {c['width']}x{c['height']} omni -> 2 x {c['pano_cols']}-wide panoramas, "
                        f"{c['feat']} ORB features/view in 12 azimuth buckets, {c['n_hyp']} RANSAC hypotheses, score={args.score}, "
                        f"refine={args.refine}" + (", solver=p3p" if getattr(args, "solver", "arun") == "p3p" else ""),
            "frames_per_step": batch, "note": note}


# ---------------------------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------------------------
def run_gpu(args, rank, local_rank, world):
    import torch
    import torch.distributed as dist
    from vo_single_camera_sos_b200 import ops, workload

    torch.cuda.set_device(local_rank)
    if world > 1:
        # NCCL may print its version banner on stdout when the communicator comes up: keep stdout for the JSON line
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)
    ctx = ops.Context(local_rank)
    if args.workload in ("c3", "c4"):
        res = (run_c3(args, ctx, rank, world, n_frames=args.frames, batch=args.batch, out_dir=args.out_dir) if args.workload == "c3"
               else run_c4(args, ctx, rank, world, steps=max(args.steps, 1) if args.steps_given else 20, warm=args.warmup))
        if rank == 0:
            res.update({"steps": args.steps, "warmup": args.warmup, "vs_baseline": None, "data": "synthetic",
                        "dtype": "u8 / f32 / f64 (as the c2 line)" if args.workload == "c3" else "f32 scoring, f64 guard path"})
            print(json.dumps(res), flush=True)
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return
    B, K, W = args.batch, args.steps, args.warmup
    n_sets = 2
    score = ops.SCORE_BEARING if args.score == "bearing" else ops.SCORE_EUCLID
    # weak scaling: every rank gets the SAME synthetic batches (seed 0), so per-GPU work is exactly what the 1-GPU run does;
    # with per-rank scenes the slowest scene, not the hardware, set the N-GPU time (3.51 vs 3.76 ms between two ranks)
    w = workload.build(ctx, args.workload, batch=B, n_frames=n_sets * B + 1, seed=0, score_mode=score,
                       solver=ops.SOLVER_P3P if args.solver == "p3p" else ops.SOLVER_ARUN, moving_fraction=args.moving)
    w.cfg.refit = {"none": ops.REFINE_NONE, "arun": ops.REFINE_ARUN, "lm": ops.REFINE_LM}[args.refine]
    c = workload.CONFIGS[args.workload]
    renderer = workload.DeviceRenderer(ctx, w)
    sets = [workload.make_frames(w, s * B, B, renderer=renderer) for s in range(n_sets)]
    dev_sets = [workload.to_device(ctx, fr) for fr in sets]
    pin_sets = [workload.to_pinned(fr) for fr in sets]
    in_bytes = sum(int(t.numel() * t.element_size()) for t in dev_sets[0])
    fe = w.frontend(ctx)
    ctx_sm_count = torch.cuda.get_device_properties(local_rank).multi_processor_count

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident throughput ---------------------------------------------------------------------------------
    for i in range(max(W, n_sets)):
        fe.step(*dev_sets[i % n_sets])
    torch.cuda.synchronize()
    sampler = ClockSampler(local_rank)
    sampler.start()
    barrier()
    launches0 = ctx.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(K):
        fe.step(*dev_sets[i % n_sets])
    e1.record()
    barrier()
    ms_dev = e0.elapsed_time(e1)
    launches = ctx.launch_count - launches0
    clocks = sampler.stop()
    stats = fe.buffers()["stats"].cpu().numpy()
    if args.dump_outputs and rank == 0:
        dump_outputs(fe.buffers(), args.dump_outputs)

    # ---- end to end: pinned host buffers in, poses out, copies overlapped with the previous step's kernels -----------
    fe2 = w.frontend(ctx)
    for i in range(max(W, n_sets)):
        fe2.step_host(*pin_sets[i % n_sets])
    barrier()
    t0 = time.perf_counter()
    prev = None
    for i in range(K):
        tk = fe2.submit_host(*pin_sets[i % n_sets])
        if prev is not None:
            fe2.wait_host(prev)
        prev = tk
    poses, st2 = fe2.wait_host(prev)
    torch.cuda.synchronize()
    ms_e2e = (time.perf_counter() - t0) * 1e3
    barrier()
    d2h_bytes = int(poses.nbytes + st2.nbytes)
    h2d_bytes, d2h_check = fe2.host_bytes()   # what submit_host actually uploads: only the LUT-reachable image bytes
    assert d2h_check == d2h_bytes
    # the ceiling of the end-to-end path: the same number of bytes as ONE plain pinned -> device copy per step, no kernels,
    # all ranks at once (what the host and the PCIe links can feed; the front-end cannot be faster than this)
    probe_src = torch.empty(h2d_bytes, dtype=torch.uint8).pin_memory()
    probe_dst = torch.empty(h2d_bytes, dtype=torch.uint8, device="cuda")
    for _ in range(2):
        probe_dst.copy_(probe_src, non_blocking=True)
    barrier()
    t0 = time.perf_counter()
    for _ in range(max(K // 4, 8)):
        probe_dst.copy_(probe_src, non_blocking=True)
    torch.cuda.synchronize()
    ms_probe = (time.perf_counter() - t0) * 1e3 / max(K // 4, 8)
    barrier()
    del probe_src, probe_dst

    # ---- per-kernel times (CUDA events after every launch, eager replays of the same steps) --------------------------
    fe.profile_begin()
    for i in range(K):
        fe.step(*dev_sets[i % n_sets])
    marks = fe.profile_end(max_n=64 * K + 64)
    torch.cuda.synchronize()
    buf = fe.buffers()
    per_step = buf["launches_per_step"]
    kernels = summarize_kernels(marks, K)
    # work actually done per step (device-side sizes)
    st_pairs = int((buf["st_q_len"].long() * buf["st_t_len"].long()).sum())
    tm_pairs = int((buf["tm_q_len"].long() * buf["tm_t_len"].long()).sum())
    n_corr = buf["n_corr"].cpu().numpy().astype(np.int64)
    rows, cols = w.cfg.pano_rows, w.cfg.pano_cols
    remap_bytes = B * (2 * rows * cols * (8 + 3) + c["height"] * c["width"] * 3)
    flop_pair = 30.0 if args.score == "euclid" else 45.0          # SURVEY 8d's model
    # executed per pair, counted in the SASS of score_kernel's inner loop (8 pairs per trip): bearing 68 FFMA2 + 8 FMUL2 =
    # 17 FFMA + 2 FMUL = 36 FLOP; euclid 52 FFMA2 + 12 FADD2 + 4 FMUL2 = 13 FFMA + 3 FADD + 1 FMUL = 30 FLOP
    flop_exec = 30.0 if args.score == "euclid" else 36.0
    popc_peak = ctx.peak_popc()   # T POPC/s, measured on this GPU just now
    ffma_peak = ctx.peak_ffma()   # TFLOP/s, measured
    peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))) if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")) else {}
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    hbm_src = "MEASURED_PEAKS.json (sustained copy)" if peaks else "fallback 6650 GB/s"

    def k_ms(name):
        return kernels.get(name, {}).get("ms", float("nan"))

    tmem_peak = ctx.peak_tmem_read()     # TB/s, measured: tcgen05.ld over all SMs
    ffma2_peak = ctx.peak_ffma2()        # TFLOP/s, measured: packed fma.rn.f32x2
    remap_name = "remap3b_kernel" if f"remap3b_kernel#0" in kernels else "remap3p_kernel"
    mma_engine = f"hamming_mma_kernel#1" in kernels
    roof = {}
    t = k_ms(f"{remap_name}#0")
    lut_bytes = 2 * rows * cols * 8
    src_reach = int(fe2.host_bytes()[0] // B - (2 * w.cfg.max_feat_per_view * (8 + 32) + 2 * (w.cfg.n_buckets + 1) * 4))
    honest = B * (2 * rows * cols * 3 + src_reach) + lut_bytes
    roof["remap"] = {"kernel": remap_name, "bound": "hbm", "achieved": honest / (t * 1e-3) / 1e9, "peak": hbm_peak,
                     "unit": "GB/s", "frac": honest / (t * 1e-3) / 1e9 / hbm_peak, "ms": t, "peak_source": hbm_src,
                     "algorithmic_bytes": honest, "traffic": None,
                     "bytes_model": "per step: panoramas out (2 x rows x cols x 3 per frame) + the LUT-reachable bytes of each omni "
                                    "image (what submit_host uploads) + the packed LUT ONCE (it is shared by all frames and stays in L2)",
                     "survey_8d_bytes": remap_bytes, "survey_8d_frac": remap_bytes / (t * 1e-3) / 1e9 / hbm_peak}
    for tag, idx, pairs in (("stereo", 0, st_pairs), ("temporal", 1, tm_pairs)):
        if mma_engine and f"hamming_mma_kernel#{idx}" in kernels:
            t = k_ms(f"hamming_mma_kernel#{idx}")
            # int8 tensor peak: 8192 MAC/clk/SM (M128 N128 K32 per 64 clk: the rate ncu's sm__pipe_tensor_cycles_active counts
            # against) at the SM clock seen during the run; no measured int8 figure exists in MEASURED_PEAKS.json, so the bf16
            # figures are shown beside it (int8 = 2 x bf16 nominal)
            sm_clk = (clocks.get("sm_mhz") or 1965.0) * 1e6
            tensor_peak = ctx_sm_count * 8192 * 2 * sm_clk / 1e12
            tops = pairs * 288.0 * 2.0 / (t * 1e-3) / 1e12
            roof[f"hamming_{tag}"] = {
                "kernel": "hamming_mma_kernel (tcgen05.mma kind::i8 + tcgen05.ld epilogue)", "bound": "tensor", "achieved": tops,
                "peak": tensor_peak, "unit": "TOP/s (int8)", "frac": tops / tensor_peak, "ms": t,
                "peak_source": "148 SMs x 8192 int8 MAC/clk x SM clock (the tensor-pipe rate; ncu sm__pipe_tensor_cycles_active "
                               "of the same kernel: profiles/r02/hamming_mma_*_metrics.txt); MEASURED_PEAKS bf16 "
                               f"{peaks.get('bf16_tflops')} TFLOP/s burst for scale",
                "descriptor_pairs": pairs, "matches_per_s": pairs / (t * 1e-3), "traffic": None,
                "algorithmic_ops_per_pair": "288 int8 MACs (256 sign products + 32 bookkeeping columns)",
                "tmem_read_tb_per_s": pairs * 4.0 / (t * 1e-3) / 1e12, "tmem_read_peak_tb_per_s": tmem_peak,
                "popc_equivalent": {"achieved_tpopc": 8.0 * pairs / (t * 1e-3) / 1e12, "peak": popc_peak,
                                    "frac": 8.0 * pairs / (t * 1e-3) / 1e12 / popc_peak},
                "expand_ms": k_ms(f"hamming_expand_kernel#{2 * idx}") + k_ms(f"hamming_expand_kernel#{2 * idx + 1}"),
                "note": "achieved counts the MACs of the REAL descriptor pairs (padding of ragged tiles excluded); popc_equivalent = "
                        "SURVEY 8d's 8-POPC-per-pair count over the POPC-pipe peak, for comparison with the integer-pipe engine"}
        else:
            t = k_ms(f"hamming_partial_kernel#{idx}")
            ops_t = 8.0 * pairs
            roof[f"hamming_{tag}"] = {
                "kernel": "hamming_partial_kernel (XOR + POPC)", "bound": "int-pipe (POPC)", "achieved": ops_t / (t * 1e-3) / 1e12,
                "peak": popc_peak, "unit": "TPOPC/s", "frac": ops_t / (t * 1e-3) / 1e12 / popc_peak * 5.0 / 8.0, "ms": t,
                "peak_source": "POPC microbenchmark run in this process", "descriptor_pairs": pairs,
                "matches_per_s": pairs / (t * 1e-3), "traffic": None, "executed_popc_per_pair": 5,
                "algorithmic_frac": ops_t / (t * 1e-3) / 1e12 / popc_peak,
                "note": "frac = share of the POPC pipe actually used (the kernel executes 5 POPC per pair after three carry-save "
                        "adders); algorithmic_frac counts SURVEY 8d's 8 POPC32 per pair and can exceed 1"}
    pairs_hc = float(w.cfg.n_hyp) * float(n_corr.sum())
    fl = pairs_hc * flop_pair
    if "score_mma_kernel#0" in kernels:
        # bearing score on the tensor cores (csrc/score_mma.cuh): 144 bf16 MACs per (hypothesis, correspondence) pair — 12 + 10
        # features x 6 partial products of the three-way bfloat16 split, zero padded to 80 + 64 K columns
        t = k_ms("score_mma_kernel#0")
        bf16_peak = float(peaks.get("bf16_tflops", 1694.3))
        mac_flop = pairs_hc * 144.0 * 2.0
        roof["ransac_score"] = {
            "kernel": "score_mma_kernel (tcgen05.mma kind::f16, bf16 x 3 split, fp32 accumulators in TMEM)", "bound": "tensor",
            "achieved": mac_flop / (t * 1e-3) / 1e12, "peak": bf16_peak, "unit": "TFLOP/s", "frac": mac_flop / (t * 1e-3) / 1e12 / bf16_peak,
            "ms": t, "peak_source": "MEASURED_PEAKS.json bf16_tflops (cuBLAS burst)" if peaks else "fallback 1694.3 TFLOP/s",
            "hypothesis_point_pairs": pairs_hc, "traffic": None, "expand_ms": k_ms("score_expand_kernel#0"),
            "algorithmic_flop_per_pair": "288 (144 bf16 MACs: the float32 products of SURVEY 8d's 45-FLOP model, each split into six bf16 products)",
            "fp32_equivalent": {"flop_per_pair_model": flop_pair, "tflops": fl / (t * 1e-3) / 1e12, "ffma_peak_tflops": ffma_peak,
                                "frac_of_fp32_peak": fl / (t * 1e-3) / 1e12 / ffma_peak,
                                "note": "SURVEY 8d's FP32-pipe count of the same work over the measured FFMA peak; above the FP32-pipe "
                                        "kernel's 0.82 because the products left that pipe"},
            "note": "the tensor pipe is NOT what limits this kernel (ncu sm__pipe_tensor_cycles_active 26 %): the epilogue is — "
                    "4 KB of accumulators per warp and tile through tcgen05.ld plus 5 ALU/FMA instructions per pair on 8 warps "
                    "(profiles/r02/score_mma_*_metrics.txt, DESIGN.md section 5)"}
    else:
        t = k_ms("score_kernel#0")
        fl_exec = pairs_hc * flop_exec
        roof["ransac_score"] = {"kernel": "score_kernel", "bound": "fp32-fma", "achieved": fl_exec / (t * 1e-3) / 1e12, "peak": ffma2_peak,
                                "unit": "TFLOP/s", "frac": fl_exec / (t * 1e-3) / 1e12 / ffma2_peak, "ms": t,
                                "peak_source": "packed fma.rn.f32x2 microbenchmark run in this process (the instruction the kernel issues); "
                                               "scalar FFMA peak beside it", "ffma_scalar_peak_tflops": ffma_peak,
                                "flop_per_pair_executed": flop_exec, "flop_per_pair_model": flop_pair,
                                "model_frac": fl / (t * 1e-3) / 1e12 / ffma_peak,
                                "note": "achieved = FLOPs the kernel executes (SASS count of the inner loop x pairs); ncu "
                                        "sm__pipe_fma_cycles_active of the same kernel: profiles/r02/score_*_metrics.txt",
                                "hypothesis_point_pairs": pairs_hc, "traffic": None}
    t = k_ms("stereo_geometry_kernel#0") + k_ms("stereo_compact_kernel#0")
    lt_bytes = 53.0 * float(buf["st_pair_count"].sum())
    roof["lift_triangulate"] = {"kernel": "stereo_geometry_kernel + stereo_compact_kernel", "bound": "hbm", "achieved": lt_bytes / (t * 1e-3) / 1e9,
                                "peak": hbm_peak, "unit": "GB/s", "frac": lt_bytes / (t * 1e-3) / 1e9 / hbm_peak, "ms": t,
                                "traffic": None}
    # DRAM traffic per launch from the committed ncu --set full captures (same workload and batch only)
    tpath = os.path.join(ROOT, "profiles", "r02", "traffic.json")
    if os.path.exists(tpath):
        tr = json.load(open(tpath))
        if tr.get("workload") == args.workload and tr.get("batch") == B:
            for k in roof:
                if k in tr:
                    roof[k]["traffic"] = tr[k]
                    roof[k]["traffic_source"] = "profiles/r02/traffic.json (ncu dram__bytes_read+write per launch)"
    dominant = max((k for k in roof if not math.isnan(roof[k]["ms"])), key=lambda k: roof[k]["ms"])

    # ---- reduce over ranks -------------------------------------------------------------------------------------------
    print(f"[bench rank {rank}] device-resident {ms_dev / K:.4f} ms/step, e2e {ms_e2e / K:.4f} ms/step, clocks {clocks}",
          file=sys.stderr, flush=True)
    if world > 1:
        tt = torch.tensor([ms_dev, ms_e2e, ms_probe], dtype=torch.float64, device="cuda")
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms_dev, ms_e2e, ms_probe = float(tt[0]), float(tt[1]), float(tt[2])
        ll = torch.tensor([launches], dtype=torch.int64, device="cuda")
        dist.all_reduce(ll, op=dist.ReduceOp.SUM)
        launches = int(ll[0])
    value = world * B * K / (ms_dev * 1e-3)
    e2e = world * B * K / (ms_e2e * 1e-3)

    cpu_base = None
    if rank == 0 and world == 1 and not args.no_cpu:
        cpu_base = cpu_baseline(args)
    refine_evals = buf["refine_stats"][:, 2].cpu().numpy().astype(int).tolist() if args.refine == "lm" else None
    corr = np.maximum(stats[:, 1].astype(np.float64), 1.0)
    inlier_ratio = float(np.median(stats[:, 2] / corr))
    fe.close(); fe2.close()
    del buf
    # the clean static scene (every landmark rigid, ~99 % inliers) as a second line: same kernels, lighter exact-path load
    clean = None
    if args.moving > 0 and not args.no_extras:
        w0 = workload.build(ctx, args.workload, batch=B, n_frames=n_sets * B + 1, seed=0, score_mode=score,
                            solver=ops.SOLVER_P3P if args.solver == "p3p" else ops.SOLVER_ARUN, moving_fraction=0.0)
        w0.cfg.refit = w.cfg.refit
        sets0 = [workload.to_device(ctx, workload.make_frames(w0, s_ * B, B, renderer=renderer)) for s_ in range(n_sets)]
        fe0 = w0.frontend(ctx)
        for i in range(max(W, n_sets)):
            fe0.step(*sets0[i % n_sets])
        barrier()
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        c0.record()
        for i in range(K):
            fe0.step(*sets0[i % n_sets])
        c1.record()
        barrier()
        ms0 = torch.tensor([c0.elapsed_time(c1)], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(ms0, op=dist.ReduceOp.MAX)
        st0 = fe0.buffers()["stats"].cpu().numpy()
        clean = {"value": world * B * K / (float(ms0[0]) * 1e-3), "unit": UNIT, "ms_per_step": float(ms0[0]) / K,
                 "median_inlier_ratio": float(np.median(st0[:, 2] / np.maximum(st0[:, 1], 1))),
                 "note": "same configuration with a static scene (--moving 0): the round-1 input set"}
        fe0.close()
        del sets0
    # BASELINE configs 3 and 4 ride along (all ranks take part): the sharded 1000-frame sequence and the split RANSAC
    extras = {}
    if not args.no_extras:
        del dev_sets, pin_sets, sets
        torch.cuda.empty_cache()
        extras["config4"] = run_c4(args, ctx, rank, world)
        extras["config3"] = run_c3(args, ctx, rank, world, n_frames=args.frames, batch=32, out_dir=args.out_dir)

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms_dev / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8 (remap, Hamming) / f32 (RANSAC scoring, f64 guard path) / f64 (lifting, 3-point Arun)",
            "data": "synthetic",
            "config": dict(workload_config(args, c, B, note=f"inputs resident in HBM; {n_sets} input sets of {in_bytes / 1e6:.0f} MB "
                                                           f"rotated (each larger than the 126 MB L2: no L2 flush needed); "
                                                           f"CUDA-graph replay of {per_step} launches per step"),
                           input_bytes_per_step=in_bytes, parallelism=f"frame batches sharded over {world} GPU(s), no collective; every rank runs the same synthetic batches"),
            "e2e": {"value": e2e, "unit": UNIT, "ms_per_step": ms_e2e / K, "h2d_bytes_per_step": h2d_bytes,
                    "d2h_bytes_per_step": d2h_bytes, "host_input_bytes_per_step": in_bytes,
                    "h2d_only_probe": {"ms_per_step": ms_probe, "gb_per_s_per_gpu": h2d_bytes / (ms_probe * 1e-3) / 1e9,
                                       "frame_pairs_per_s_ceiling": world * B / (ms_probe * 1e-3),
                                       "note": "one plain pinned->device copy of h2d_bytes_per_step per step on every rank at "
                                               "once, no kernels (max over ranks): the feed ceiling of the host/PCIe path"},
                    "note": "sos_frontend_submit_host/wait_host on pinned host buffers, 2 staging slots (copies overlap kernels); "
                            "of each omni image only the bytes the panoramic LUT can read are uploaded (row bands)"},
            "gpu_launches": launches,
            "roofline": dict(roof[dominant], name=dominant),
            "roofline_hbm": dict(roof["remap"], name="remap"),
            "kernels": roof,
            "kernel_ms_per_step": {k: round(v["ms"], 4) for k, v in sorted(kernels.items(), key=lambda kv: -kv[1]["ms"])},
            "hamming_matches_per_s": (st_pairs + tm_pairs) / ((roof["hamming_stereo"]["ms"] + roof["hamming_temporal"]["ms"]) * 1e-3),
            "hamming_engine": "tcgen05 int8 (hamming_mma_kernel)" if mma_engine else "XOR+POPC (hamming_partial_kernel)",
            "cpu_baseline": cpu_base,
            "clocks": clocks,
            "stats_last_step": {"stereo_correspondences": stats[:, 0].tolist(), "temporal_correspondences": stats[:, 1].tolist(),
                                "ransac_inliers": stats[:, 2].tolist(), "median_inlier_ratio": inlier_ratio,
                                "moving_landmark_share": args.moving, "refine_evaluations": refine_evals},
            "clean_scene": clean,
            "config3": extras.get("config3"), "config4": extras.get("config4"),
            "peaks": {"hbm_gbs": hbm_peak, "popc_tera_per_s": popc_peak, "ffma_tflops": ffma_peak, "ffma2_tflops": ffma2_peak,
                      "tmem_read_tb_per_s": tmem_peak},
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


# ---------------------------------------------------------------------------------------------------------------------
# BASELINE config 3: one 1000-frame sequence, frame pairs sharded over the ranks (strong scaling, no data-path collective)
# ---------------------------------------------------------------------------------------------------------------------
def run_c3(args, ctx, rank, world, n_frames=1000, batch=32, geometry="c1", out_dir=None):
    import torch
    import torch.distributed as dist
    from vo_single_camera_sos_b200 import ops, sequence, workload

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    w = workload.build(ctx, geometry, batch=batch, n_frames=n_frames, seed=0, score_mode=ops.SCORE_BEARING)
    plan = sequence.plan_shard(n_frames, world, rank, batch)
    counts = [sequence.plan_shard(n_frames, world, r, batch) for r in range(world)]
    omni = workload.DeviceRenderer(ctx, w).render(w.trajectory[0]).cpu().numpy()
    t_gen = time.perf_counter()
    batches = sequence.make_shard_batches(w, plan, batch, omni=omni)
    t_gen = time.perf_counter() - t_gen
    fe = w.frontend(ctx)
    h2d, d2h = fe.host_bytes()
    for _ in range(2):                                   # warm-up: graph capture, arena sizing, staging buffers
        sequence.run_shard(fe, batches[:2], sequence.ShardPlan(plan.first, plan.first, plan.read_first, 0), batch)
    barrier()
    l0 = ctx.launch_count
    t0 = time.perf_counter()
    rel, stats = sequence.run_shard(fe, batches, plan, batch)
    torch.cuda.synchronize()
    t_rank = time.perf_counter() - t0
    launches = ctx.launch_count - l0
    pose_all = sequence.gather_to_rank0(torch.from_numpy(rel).cuda(), [c.last - c.first for c in counts])
    stat_all = sequence.gather_to_rank0(torch.from_numpy(stats).cuda(), [c.last - c.first for c in counts])
    traj = failed = None
    if rank == 0:
        rel_all, st_all = pose_all.cpu().numpy(), stat_all.cpu().numpy()
        traj, failed = sequence.chain_trajectory(rel_all, st_all)
    barrier()
    t_all = time.perf_counter() - t0
    tt = torch.tensor([t_rank, t_all], dtype=torch.float64, device="cuda")
    ll = torch.tensor([launches], dtype=torch.int64, device="cuda")
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dist.all_reduce(ll, op=dist.ReduceOp.SUM)
    res = None
    if rank == 0:
        # every shard boundary pair (f-1 on one rank's block, f on the next) recomputed on this GPU as a two-frame shard:
        # must be bit-identical to what the owning rank returned (the one-frame overlap works)
        same = True
        for r in range(1, world):
            f = counts[r].first
            if counts[r].last <= f:
                continue
            mini = sequence.ShardPlan(f, f + 1, f - 1, 1)
            p2, s2 = sequence.run_shard(fe, sequence.make_shard_batches(w, mini, batch, omni=omni), mini, batch)
            same = same and np.array_equal(p2[0], rel_all[f]) and np.array_equal(s2[0], st_all[f])
        gt = np.linalg.inv(w.trajectory[0]) @ w.trajectory[n_frames - 1]
        end_err = float(np.linalg.norm(traj[-1][:3, 3] - gt[:3, 3]))
        gt_rel = np.linalg.inv(w.trajectory[:-1]) @ w.trajectory[1:]
        pair_t_err = np.linalg.norm(rel_all[1:, :, 3] - gt_rel[:, :3, 3], axis=1)
        dR = np.einsum("nij,nkj->nik", rel_all[1:, :, :3].astype(np.float64), gt_rel[:, :3, :3])
        pair_r_err = np.degrees(np.arccos(np.clip(0.5 * (np.trace(dR, axis1=1, axis2=2) - 1.0), -1.0, 1.0)))
        path = float(sum(np.linalg.norm((np.linalg.inv(w.trajectory[i]) @ w.trajectory[i + 1])[:3, 3]) for i in range(n_frames - 1)))
        if out_dir:
            os.makedirs(out_dir, exist_ok=True)
            sequence.write_tum(os.path.join(out_dir, f"c3_estimated_frame_poses_TUM_{world}gpu.txt"), traj)
        c = workload.CONFIGS[geometry]
        res = {
            "metric": "sos_sequence_frames_per_s", "value": n_frames / float(tt[1]), "unit": "frames/s", "n_gpus": world,
            "scaling": "strong", "higher_is_better": True, "seconds": float(tt[1]), "seconds_slowest_rank_shard": float(tt[0]),
            "config": {"workload": f"c3: {n_frames}-frame synthetic SOS sequence, {geometry} geometry ({c['width']}x{c['height']} omni, "
                                   f"{c['feat']} features/view, {c['n_hyp']} hypotheses), consecutive frame pairs, batches of {batch}",
                       "parallelism": f"contiguous blocks of frames per rank with one overlapping frame ({world} rank(s)); "
                                      "no data-path collective; relative poses (48 B per pair) gathered to rank 0 and chained there",
                       "timed": "pinned host inputs -> sos_frontend_submit_host/wait_host per batch -> gather -> trajectory on rank 0"},
            "e2e_bytes": {"h2d_bytes_per_batch": h2d, "d2h_bytes_per_batch": d2h},
            "gpu_launches": int(ll[0]), "frames_per_rank": [c_.last - c_.first for c_ in counts],
            "trajectory_sha256": sequence.trajectory_digest(rel_all, st_all),
            "boundary_pairs_identical_to_local_recompute": bool(same), "pairs_failed": len(failed),
            "end_position_error_m": end_err, "path_length_m": path,
            "pair_translation_error_median_m": float(np.median(pair_t_err)), "pair_rotation_error_median_deg": float(np.median(pair_r_err)),
            "drift_note": "frame-to-frame chaining of 999 relative poses, no keyframes: the end error is accumulated drift of the "
                          "synthetic measurement noise (0.15 px), not a parity figure",
            "median_inliers": float(np.median(st_all[1:, 2])), "feature_synthesis_s_rank0": t_gen,
        }
    fe.close()
    return res


# ---------------------------------------------------------------------------------------------------------------------
# BASELINE config 4: one huge RANSAC, hypotheses split over the ranks, winners combined by one 8-byte NCCL MAX
# ---------------------------------------------------------------------------------------------------------------------
def c4_problem(n=50000, H=65536, seed=4):
    rng = np.random.default_rng(seed)   # same data on every rank: the correspondences are replicated (1.2 MB)
    p_cur = rng.normal(size=(1, n, 3))
    p_cur = (p_cur / np.linalg.norm(p_cur, axis=2, keepdims=True) * rng.uniform(0.5, 7.0, (1, n, 1))).astype(np.float32)
    ang = np.deg2rad(2.0)
    R = np.array([[np.cos(ang), -np.sin(ang), 0], [np.sin(ang), np.cos(ang), 0], [0, 0, 1]], np.float32)
    p_ref = (p_cur @ R.T + np.float32([0.03, -0.01, 0.02]) + rng.normal(0, 0.005, p_cur.shape)).astype(np.float32)
    out = rng.random(n) > 0.35          # 35 % inliers (the reference's assumed outlier fraction 0.65, pose_est_tools.py:675)
    p_ref[0, out] = (rng.normal(size=(int(out.sum()), 3)) * 3).astype(np.float32)
    hyp = rng.integers(0, 2 ** 32, (H, 3), dtype=np.uint64).astype(np.uint32)
    return p_ref, p_cur, hyp


def run_c4(args, ctx, rank, world, steps=20, warm=3):
    import torch
    import torch.distributed as dist
    from vo_single_camera_sos_b200 import ops, parallel
    n, H = 50000, 65536
    p_ref, p_cur, hyp = c4_problem(n, H)
    d = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    P_ref, P_cur, N = d(p_ref), d(p_cur), torch.tensor([n], dtype=torch.int32, device="cuda")
    hyp_d = d(hyp.view(np.int32))
    run = lambda: parallel.ransac_split(ctx, P_ref, P_cur, N, hyp_d, ops.SCORE_EUCLID, 0.05)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(warm):
        res = run()
    barrier()
    l0 = ctx.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        res = run()
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1) / steps
    launches = ctx.launch_count - l0
    # the collective's share: the same 8-byte all-reduce alone, back to back, on the same stream
    ar_ms = 0.0
    if world > 1:
        key = torch.zeros(1, dtype=torch.int64, device="cuda")
        for _ in range(5):
            dist.all_reduce(key, op=dist.ReduceOp.MAX)
        torch.cuda.synchronize()
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record()
        for _ in range(50):
            dist.all_reduce(key, op=dist.ReduceOp.MAX)
        a1.record()
        torch.cuda.synchronize()
        ar_ms = a0.elapsed_time(a1) / 50
    tt = torch.tensor([ms, ar_ms], dtype=torch.float64, device="cuda")
    ll = torch.tensor([launches], dtype=torch.int64, device="cuda")
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dist.all_reduce(ll, op=dist.ReduceOp.SUM)
    out = None
    if rank == 0:
        pose, count, mask, winner = res
        fp, fh, fc, fm, _ = ctx.ransac_p3d(P_ref, P_cur, N, hyp_d, ops.SCORE_EUCLID, 0.05)   # the undivided list on this GPU
        verified = bool(int(fh[0]) == int(winner[0]) and int(fc[0]) == int(count[0]) and torch.equal(fm, mask)
                        and torch.equal(fp, pose))
        pairs = float(n) * H
        ffma = ctx.peak_ffma2()
        tfl = pairs * 30 / (float(tt[0]) * 1e-3) / 1e12
        out = {
            "metric": "ransac_hypothesis_point_pairs_per_s", "value": pairs / (float(tt[0]) * 1e-3), "unit": "pairs/s",
            "n_gpus": world, "steps": steps, "warmup": warm, "ms_per_step": float(tt[0]), "higher_is_better": True,
            "scaling": "strong",
            "config": {"workload": f"c4: {n} 3D-3D correspondences x {H} hypotheses, euclid score, 35 % inliers",
                       "parallelism": f"hypothesis list split over {world} rank(s); one int64 MAX all-reduce per step (NCCL), "
                                      "then every rank re-derives the winner's pose and inlier mask locally"},
            "allreduce_ms": float(tt[1]), "allreduce_share": float(tt[1]) / float(tt[0]) if world > 1 else 0.0,
            "winner": int(winner[0]), "inliers": int(count[0]), "matches_single_gpu_full_list": verified,
            "gpu_launches": int(ll[0]),
        }
        if os.environ.get("SOS_SCORE_ENGINE", "")[:1] == "f":
            out["roofline"] = {"bound": "fp32-fma", "achieved": tfl, "peak": ffma * world, "unit": "TFLOP/s", "frac": tfl / (ffma * world),
                               "note": "score_kernel: 30 FLOP per (hypothesis, correspondence) executed (SASS count; equals SURVEY 8d's "
                                       "model) over all ranks; peak = packed-FMA microbenchmark x ranks"}
        else:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))) if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")) else {}
            bf16 = float(peaks.get("bf16_tflops", 1694.3))
            mac = pairs * 144.0 * 2.0 / (float(tt[0]) * 1e-3) / 1e12
            out["roofline"] = {"bound": "tensor", "achieved": mac, "peak": bf16 * world, "unit": "TFLOP/s", "frac": mac / (bf16 * world),
                               "note": "score_mma_kernel (Euclidean score as two bfloat16-split GEMMs, csrc/score_mma.cuh): 144 bf16 MACs per "
                                       "(hypothesis, correspondence) over the WHOLE step (hypothesis generation, expansion, deferred "
                                       "re-decisions and the winner's re-derivation included); peak = MEASURED_PEAKS bf16 x ranks",
                               "fp32_equivalent_tflops": tfl, "ffma_peak_tflops": ffma * world}
    return out


DUMP_ARRAY_BYTES = 16 << 20   # per array: the six arrays stay under 64 MB in all


def dump_outputs(buf, out_dir):
    """Write what the last step computed, as a caller of Frontend.step reads it from buffers(), to out_dir/<name>.npy: per
    frame pair the refitted pose, RANSAC's pose, the stats row (stereo points, correspondences, inliers, winning hypothesis),
    the inlier mask over the correspondences and the triangulated stereo points of the new frame, and the panoramas.  Rows
    past a frame's valid count are zeroed, since they hold whatever an earlier step left there.  int32 goes out as float64,
    the rest as float32 (both exact).  An array above DUMP_ARRAY_BYTES is replaced by a fixed, seeded sample of its elements
    (flattened, in index order), so the same arguments give the same files from run to run."""
    import torch
    B = buf["pose"].shape[0]

    def valid(t, n):
        keep = torch.arange(t.shape[1], device=t.device)[None, :] < n[:, None]
        return torch.where(keep.view(keep.shape + (1,) * (t.dim() - 2)), t, torch.zeros((), dtype=t.dtype, device=t.device))

    arrays = {"pose": buf["pose"], "ransac_pose": buf["ransac_pose"], "stats": buf["stats"],
              "inlier_mask": valid(buf["inlier_mask"], buf["n_corr"]),
              "points": valid(buf["xyz"][1:B + 1], buf["n"][1:B + 1]),   # slot i + 1 holds frame i of the batch
              "panoramas": buf["pano"]}
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        dtype = torch.float64 if t.dtype == torch.int32 else torch.float32
        size = 8 if dtype == torch.float64 else 4
        if t.numel() * size > DUMP_ARRAY_BYTES:
            idx = np.sort(np.random.default_rng(0).choice(t.numel(), DUMP_ARRAY_BYTES // size, replace=False))
            t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
        np.save(os.path.join(out_dir, f"{name}.npy"), t.to(dtype).cpu().numpy())


def summarize_kernels(marks, steps):
    """marks: (kernel name, ms) per launch over `steps` eager steps -> average ms per step, keyed `kernel#k` for the k-th
    launch of that kernel within a step (e.g. hamming_mma_kernel#0 = stereo buckets, #1 = temporal matching)."""
    per = len(marks) // steps
    out = {}
    for s in range(steps):
        seen = {}
        for name, ms in marks[s * per:(s + 1) * per]:
            k = seen.get(name, 0)
            seen[name] = k + 1
            out.setdefault(f"{name}#{k}", []).append(ms)
    return {k: {"ms": sum(v) / len(v), "n": len(v)} for k, v in out.items()}


def cpu_baseline(args):
    n_pairs = 3 if args.workload == "c2" else 6
    cpu = CpuPath(args.workload, seed=0, n_frames=n_pairs + 2, score_mode=args.score, refine=args.refine, moving=args.moving)
    cpu.prime()
    cpu.pair()  # warm-up (OpenCV thread pool, NumPy caches)
    cpu.timer.clear()
    t0 = time.perf_counter()
    inl = []
    for _ in range(n_pairs):
        o = cpu.pair()
        inl.append((o["best_count"], o["n_corr"]) if o else (-1, 0))
    dt = time.perf_counter() - t0
    stages = {k: round(v / n_pairs, 4) for k, v in cpu.timer.items()}
    # the same pairs with the reference's own RANSAC budget (210 iterations, pose_est_tools.py:675-676, 709-720)
    cpu2 = CpuPath(args.workload, seed=0, n_frames=n_pairs + 2, score_mode=args.score, refine=args.refine, moving=args.moving)
    cpu2.hyp_limit = 210
    cpu2.prime()
    cpu2.timer.clear()
    t1 = time.perf_counter()
    for _ in range(n_pairs):
        cpu2.pair()
    dt2 = time.perf_counter() - t1
    return {"value": n_pairs / dt, "unit": UNIT, "cores": cpu.threads, "kind": "port", "seconds": dt,
            "seconds_per_pair_by_stage": stages,
            "ransac_share": round(cpu.timer.get("ransac", 0.0) / dt, 3),
            "value_at_reference_ransac_budget": n_pairs / dt2, "reference_ransac_budget_hypotheses": 210,
            "seconds_per_pair_by_stage_at_reference_budget": {k: round(v / n_pairs, 4) for k, v in cpu2.timer.items()},
            "inliers_of_correspondences": inl,
            "sample": f"{n_pairs} frame pairs of {args.workload} through oracle.pipeline: OpenCV calls as the reference makes "
                      f"them (cv2.getNumThreads()={cpu.threads}, os.cpu_count()={os.cpu_count()}): get_fully_masked_images incl. "
                      f"its float64 temporaries, float64->float32 LUT cast + cv2.remap, BFMatcher.match + sorted; NumPy float64 "
                      f"lifting / triangulation; RANSAC = NumPy float64 restatement over the same {cpu.c['n_hyp']} hypotheses "
                      f"(OpenGV absent: the reference hands this step to OpenGV C++ with <= 210 iterations - see "
                      f"value_at_reference_ransac_budget); 'value' is the like-for-like configuration of the GPU arm"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2", choices=["c1", "c2", "tiny", "c3", "c4"],
                    help="c2 (default, the metric's configuration), c1, tiny; c3 = 1000-frame sequence sharded over the ranks; "
                         "c4 = 50k x 65536 RANSAC split over the ranks (both also ride along with the default run)")
    ap.add_argument("--frames", type=int, default=1000, help="c3: frames in the sequence")
    ap.add_argument("--no-extras", action="store_true", help="default run only: skip the config 3 / config 4 legs")
    ap.add_argument("--out-dir", default=None, help="c3: write the estimated trajectory (TUM format) here")
    ap.add_argument("--batch", type=int, default=32, help="frames (= frame pairs) per step and GPU")
    ap.add_argument("--score", default="bearing", choices=["bearing", "euclid"])
    ap.add_argument("--refine", default="arun", choices=["none", "arun", "lm"],
                    help="pose after RANSAC: Arun refit on the inliers, or Levenberg-Marquardt on the bearing residual")
    ap.add_argument("--solver", default="arun", choices=["arun", "p3p"],
                    help="RANSAC hypotheses: 3-point Arun on 3D-3D correspondences (north_star) or the bearing-only three-point solver")
    ap.add_argument("--moving", type=float, default=0.79,
                    help="share of scene landmarks that move between frames (outliers for RANSAC): 0.79 gives the ~35 %% inlier "
                         "rate SURVEY 8d specifies for config 2; 0 = the clean static scene (~99 %% inliers)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the CPU baseline leg")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (float32 / float64, "
                         "panoramas as a fixed seeded sample, under 64 MB in all) to compare two builds output for output")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.workload in ("c3", "c4")):
        ap.error("--dump-outputs applies to the frame-pair workloads (c1, c2, tiny) of --impl ours")
    rank, local_rank, world = env_int("RANK", 0), env_int("LOCAL_RANK", 0), env_int("WORLD_SIZE", 1)
    args.steps_given = args.steps is not None
    if args.steps is None:
        args.steps = 500 if args.impl == "ours" else 5  # ~0.65 s timed region: enough nvidia-smi clock samples
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world == 1 and args.gpus > 1:
        # launched without torchrun: re-exec under torch.distributed.run
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", str(29500 + os.getpid() % 1000), os.path.abspath(__file__)] + sys.argv[1:]
        os.execv(sys.executable, cmd)
    run_gpu(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
