#!/usr/bin/env python
"""bench.py -- SparseImgAlign frames/sec on the BASELINE.json workload (C1), one process per GPU.

Workload (`config`, identical in both arms): one synthetic 640x480 camera stream per GPU, 300 features per frame,
pyramid levels 4..0, <=30 Gauss-Newton iterations per level (BASELINE.json configs[1]).  One *pass* = svo::SparseImgAlign::run
over a window of `pairs_per_step_per_gpu` consecutive frame pairs of the stream (frame k is the reference of pair k and the
current frame of pair k-1); every pair starts from the identity relative pose, so the pairs of a window are independent.  A
*step* = `passes_per_step` = ceil(500 / steps) passes, so that the timed region of EXACTLY `steps` steps spans >= 0.5 s.

Legs of a run (CUDA events on the library's stream, barrier + sync on both sides, max over ranks):
  value          pyramids + feature records resident in HBM; steps x passes launches of the alignment kernel.
  e2e            through the C ABI with HOST (pinned) buffers: every frame's level-0 image is copied host->device and its
                 pyramid built on the GPU, features are packed + copied, the kernel runs, poses / masks / counters come back.
  latency_B1     configs[1] as the reference is driven (frame_handler_mono.cpp:129-140): one pair per ABI call, pair k+1
                 after pair k returned -- device time of the launch and wall time of the call incl. the new frame's upload.
  c4_32_per_gpu  configs[4] literally: 32 pairs per GPU per launch.
  roofline_by_kernel  every kernel of the path at its BASELINE config: live device time (CUDA events inside the library)
                 against its algorithmic bytes (SURVEY.md 8d) and the measured HBM peak; DRAM traffic from the committed ncu
                 captures (profiles/r02_kernels_dram.json).
`--impl reference` times oracle/_ref (the reference's own sparse_img_align.cpp compiled in place; its build system cannot run
here: Eigen, OpenCV, Sophus, vikit, Boost are absent) on the host cores the process may use, same config, and reports the
one-thread figure beside the all-thread one with the affinity mask and cgroup quota it ran under.

L2 policy: inputs larger than L2 (3552 pairs, 3553 distinct pyramids ~ 1.45 GB of images per pass vs 126 MB of L2); no flush.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "SparseImgAlign frames/sec at 640x480/300 feats/5 lvls; pose RMSE vs ref"
UNIT = "frames/s"
W, H, NFEAT, NLEVELS, MAX_LEVEL, MIN_LEVEL, NITER = 640, 480, 300, 5, 4, 0, 30
FRAME_BYTES = 409200  # 5 pyramid levels of 640x480


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--pairs-per-gpu", type=int, default=3552)  # 8 full waves of 3 CTAs x 148 SMs
    ap.add_argument("--cpu-sample", type=int, default=256, help="pairs timed by the single-thread cpu_baseline leg")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--e2e-chunks", type=int, default=4, help="chunks of the window in the e2e leg (copy/compute overlap)")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip latency / C4 / per-kernel roofline side measurements")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed (rank 0) as DIR/<name>.npy")
    return ap.parse_args()


def make_config(args) -> dict:
    """The workload description both arms print verbatim."""
    B = args.pairs_per_gpu
    return {"workload": "C1 single stream 640x480 / 300 feats / levels 4..0 / 30 GN iters, as a window of consecutive frame pairs",
            "pairs_per_step_per_gpu": B, "passes_per_step": passes_per_step(args.steps),
            "parallelism": f"{args.gpus} independent streams (one per GPU), no collective",
            "l2_policy": "inputs larger than L2 (distinct pyramids per pair, ~%d MB per pass per GPU)" % ((B + 1) * FRAME_BYTES // 1000000),
            "pyramid_rule": "vikit x86 (SSE2 avg-of-avg where width % 16 == 0)"}


def passes_per_step(steps: int) -> int:
    return max(1, math.ceil(500 / max(steps, 1)))  # 500 launches of ~1.3 ms: >= 0.5 s on the device


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons while the timed regions run."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "50"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
                for nme, val in zip(names, r[3:7]):
                    if val.lower().startswith("active"):
                        reasons.add(nme)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def algorithmic_bytes(stats, n_feat: int) -> float:
    """Compulsory bytes of one frame pair (DESIGN.md 'algorithmic bytes'; SURVEY.md 8d adapted to this kernel's records):
    49 B ref footprint per visible patch per level, 65 B feature record once, 25 B current-image footprint per in-image patch
    per residual pass, pose in/out + H + counters + visibility mask out."""
    return (49.0 * float(stats["sum_visible"]) + 65.0 * n_feat + 25.0 * float(stats["sum_in_image"]) +
            96 + 96 + 288 + 16 + n_feat)


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir: str, res: dict):
    """The results of the timed path's last step as its caller receives them (sia_batch_fetch): relative poses T
    [pairs, 3, 4] f64, visibility mask [pairs, features] f32 and the per-pair counters f64.  Above 64 MB in all, a fixed
    seeded sample of the pairs is written, its indices in pairs.npy."""
    B = len(res["T"])
    arrays = {"T": res["T"], "visible": res["visible"].reshape(B, -1).astype(np.float32)}
    arrays.update({k: res["stats"][k].astype(np.float64) for k in res["stats"].dtype.names})
    per_pair = sum(a.nbytes for a in arrays.values()) / B + 8
    if per_pair * B > DUMP_LIMIT_BYTES:
        pairs = np.sort(np.random.default_rng(0).choice(B, int((DUMP_LIMIT_BYTES - 4096) // per_pair), replace=False))
        arrays = {k: a[pairs] for k, a in arrays.items()}  # (4 KB left for the .npy headers)
        arrays["pairs"] = pairs.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def make_inputs(seed: int, B: int, device: str):
    from rpg_svo_b200 import synth

    st = synth.make_stream_fast(seed, B + 1, W, H, NFEAT, NLEVELS, device=device)
    feats = st["feats"]
    px = np.concatenate([feats[k]["px"] for k in range(B)])
    f = np.concatenate([feats[k]["f"] for k in range(B)])
    pos = np.concatenate([feats[k]["pos"] for k in range(B)])
    hp = np.concatenate([feats[k]["has_point"] for k in range(B)])
    off = np.arange(B + 1, dtype=np.int32) * NFEAT
    ref_pos = np.stack([synth.se3_inv(st["poses"][k])[:, 3] for k in range(B)])
    T0 = np.tile(synth.se3_identity()[None], (B, 1, 1))
    T_gt = np.stack([synth.se3_mul(st["poses"][k + 1], synth.se3_inv(st["poses"][k])) for k in range(B)])
    return dict(cam=st["cam"], level0=st["level0"], px=px, f=f, pos=pos, hp=hp, off=off, ref_pos=ref_pos,
                T0=T0, T_gt=T_gt, poses=np.stack(st["poses"]))


def cpu_runner(ob, synth, inp, n: int):
    """The CPU implementation of the step's first n frame pairs: returns (kind, note, stream).
    kind "reference" = oracle/_ref, svo::SparseImgAlign::run of the reference's own svo/src/sparse_img_align.cpp + frame.cpp
    compiled in place (stand-in third-party headers, see DESIGN.md 2); "port" = the oracle restatement when oracle/_ref was
    never built."""
    sl = slice(0, n * NFEAT)
    if ob.ref_lib() is not None:
        rs = ob.RefStream(inp["level0"][:n + 1].cpu().numpy(), inp["cam"], NLEVELS, inp["poses"][:n + 1], inp["off"][:n + 1],
                          inp["px"][sl], inp["f"][sl], inp["pos"][sl], inp["hp"][sl])
        note = ("svo::SparseImgAlign::run from the reference's own svo/src/sparse_img_align.cpp + frame.cpp, compiled in "
                "place with g++ -O3 -mfma -mavx2 against stand-in Eigen/Sophus/vikit/OpenCV headers (oracle/shim); "
                "a fresh SparseImgAlign per frame as in FrameHandlerMono::processFrame; pyramids prebuilt by the reference's "
                "createImgPyramid")

        def run(n_threads, want_poses=False):
            return rs.run(n_threads, MAX_LEVEL, MIN_LEVEL, NITER, want_poses=want_poses)

        return "reference", note, run
    pyrs = [synth.build_pyramid(inp["level0"][i].cpu().numpy(), NLEVELS) for i in range(n + 1)]

    def run(n_threads, want_poses=False):
        t0 = time.perf_counter()
        ob.sparse_img_align_batch(pyrs[:n], pyrs[1:n + 1], inp["cam"], inp["T0"][:n], inp["off"][:n + 1], inp["px"][sl],
                                  inp["f"][sl], inp["pos"][sl], inp["hp"][sl], inp["ref_pos"][:n], MAX_LEVEL, MIN_LEVEL,
                                  NITER, n_threads=n_threads)
        return dict(seconds=time.perf_counter() - t0, T=None)

    return "port", "CPU oracle port of svo::SparseImgAlign::run (oracle/_ref not built on this box)", run


def run_reference(args):
    """CPU arm (rank 0 only): the reference's own SparseImgAlign (oracle/_ref) on the host cores this process may use."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    from oracle import binding as ob
    from rpg_svo_b200 import shard, synth

    ob.build()
    limits = shard.host_cpu_limits()
    threads = shard.usable_threads()
    B = args.pairs_per_gpu
    passes = passes_per_step(args.steps)
    inp = make_inputs(shard.stream_seed(0), B, "cuda" if _has_cuda() else "cpu")
    kind, note, run = cpu_runner(ob, synth, inp, B)
    for _ in range(min(args.warmup, 2)):
        run(threads)
    dt = 0.0
    for _ in range(args.steps):
        for _ in range(passes):
            dt += run(threads)["seconds"]
    fps = B * passes * args.steps / dt
    # the north_star's own denominator beside it: ONE thread, on a slice of the same window
    n1 = min(args.cpu_sample, B)
    k1, _, run1 = cpu_runner(ob, synth, inp, n1)
    run1(1)
    t1 = run1(1)["seconds"]
    line = {"impl": "reference", "metric": METRIC, "value": fps, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32/f64",
            "data": "synthetic", "config": make_config(args),
            "cpu_baseline": {"value": fps, "unit": UNIT, "cores": threads, "kind": kind,
                             "sample": f"{B} frame pairs x {passes} passes x {args.steps} steps, {threads} threads",
                             "single_thread_value": n1 / t1, "single_thread_sample": f"first {n1} pairs, 1 thread",
                             "host": limits, "note": note},
            "e2e": {"value": fps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def _has_cuda() -> bool:
    try:
        import torch

        return torch.cuda.is_available()
    except Exception:
        return False


# ---------------------------------------------------------------------------------------------------------------
# side measurements: live stream latency, configs[4], per-kernel rooflines
# ---------------------------------------------------------------------------------------------------------------
def measure_latency_and_c4(ctx, capi, torch, stream, inp, host_l0, pool) -> dict:
    """configs[1] as a live stream (B = 1 per call) and configs[4] (32 pairs per GPU)."""
    out = {}
    fr = pool.frames
    nlive = 64

    def staged_device_us(B, first, reps):
        n0, n1 = first * NFEAT, (first + B) * NFEAT
        ctx.sia_batch_stage(fr[first:first + B], fr[first + 1:first + B + 1], inp["cam"], inp["T0"][first:first + B],
                            inp["off"][first:first + B + 1] - inp["off"][first], inp["px"][n0:n1], inp["f"][n0:n1], inp["pos"][n0:n1],
                            inp["hp"][n0:n1], inp["ref_pos"][first:first + B], MAX_LEVEL, MIN_LEVEL, NITER)
        for _ in range(3):
            ctx.sia_batch_run()
        ctx.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(reps):
            ctx.sia_batch_run()
        e1.record(stream)
        ctx.synchronize()
        return 1e3 * e0.elapsed_time(e1) / reps

    # ---- B = 1: device time of one pair's launch, over 64 different pairs of the stream
    dev = np.array([staged_device_us(1, k, 20) for k in range(nlive)])
    # ---- live stream end to end: per arriving frame, upload its level 0 from pinned host memory (+ pyramid on the device), then
    #      one svo_b200_sparse_img_align call against the previous frame; pair k+1 is issued after pair k returned
    ping = [capi.Frame(ctx, W, H, NLEVELS), capi.Frame(ctx, W, H, NLEVELS)]
    base = host_l0.data_ptr()
    ping[0].upload_ptrs([base])
    ctx.synchronize()

    def live(n):
        for k in range(n):
            s = slice(k * NFEAT, (k + 1) * NFEAT)
            ping[(k + 1) & 1].upload_ptrs([base + (k + 1) * W * H])
            ctx.sparse_img_align(ping[k & 1], ping[(k + 1) & 1], inp["cam"], inp["T0"][k], inp["px"][s], inp["f"][s], inp["pos"][s],
                                 inp["hp"][s], inp["ref_pos"][k], MAX_LEVEL, MIN_LEVEL, NITER)

    live(8)
    ping[0].upload_ptrs([base]); ctx.synchronize()
    t0 = time.perf_counter(); live(nlive); t1 = time.perf_counter()
    out["latency_B1"] = {"config": "configs[1] as a live stream: one pair per ABI call, pair k+1 issued after pair k returned",
                         "device_us_per_pair": float(dev.mean()), "device_us_median": float(np.median(dev)),
                         "device_us_max": float(dev.max()), "pairs": nlive,
                         "e2e_us_per_frame": 1e6 * (t1 - t0) / nlive,
                         "e2e_includes": "pinned-host level-0 upload (307 KB) + device pyramid + feature H2D + kernel + pose/mask D2H, via python ctypes",
                         "frames_per_s_e2e": nlive / (t1 - t0),
                         "launch_geometry": "4-CTA thread-block cluster per pair, all levels prepared before the first iteration, sums exchanged by st.async + mbarrier"}
    for f_ in ping:
        f_.destroy()
    # ---- configs[4]: 32 pairs per GPU per launch
    us32 = staged_device_us(32, 0, 100)
    p32 = capi.FramePool(ctx, W, H, NLEVELS, 33)

    def e2e32():
        p32.upload(0, 33, base, W * H)
        n1 = 32 * NFEAT
        ctx.sia_batch_stage(p32.frames[:32], p32.frames[1:33], inp["cam"], inp["T0"][:32], inp["off"][:33], inp["px"][:n1], inp["f"][:n1],
                            inp["pos"][:n1], inp["hp"][:n1], inp["ref_pos"][:32], MAX_LEVEL, MIN_LEVEL, NITER)
        ctx.sia_batch_run()
        return ctx.sia_batch_fetch()

    e2e32(); e2e32()
    t0 = time.perf_counter()
    for _ in range(20):
        e2e32()
    t32 = (time.perf_counter() - t0) / 20
    p32.destroy()
    out["c4_32_per_gpu"] = {"config": "configs[4]: 256 pairs over 8 GPUs = 32 pairs per GPU per launch",
                            "device_us_per_launch": us32, "frames_per_s_device": 32 / (us32 * 1e-6),
                            "e2e_us_per_launch": 1e6 * t32, "frames_per_s_e2e": 32 / t32,
                            "launch_geometry": "4-CTA cluster per pair (upfront variant, st.async exchange), 128 CTAs"}
    return out


def measure_kernels(ctx, capi, peak_gbs: float, quick: bool = False) -> dict:
    """Every kernel of the path at its BASELINE config through the C ABI, next to oracle/_ref on one host thread (algorithm
    time only, no per-item FFI): live device time from the library's CUDA events -> achieved GB/s on the algorithmic bytes of
    SURVEY.md 8d -> fraction of the measured HBM peak.  `e2e_ms` = the whole ABI call with host buffers."""
    from oracle import binding as ob  # checker / CPU baseline only
    from rpg_svo_b200 import synth

    have_ref = ob.ref_lib() is not None
    traffic = {}
    tpath = os.path.join(ROOT, "profiles", "r02_kernels_dram.json")
    if os.path.exists(tpath):
        traffic = json.load(open(tpath))
    out = {}

    def timed(fn, reps):
        if quick:  # one launch per kernel: the ncu capture list of scripts/profile_kernels.sh
            reps = 1
        else:
            fn(); fn()
        ks, t0 = [], time.perf_counter()
        for _ in range(reps):
            fn()
            ks.append(ctx.last_kernel_ms())
        return float(np.median(ks)), 1e3 * (time.perf_counter() - t0) / reps

    def entry(name, kernel, units, unit_name, alg_bytes, k_ms, e2e_ms, cpu_ms, cpu_kind, extra=None):
        ach = alg_bytes / (k_ms * 1e-3) / 1e9
        tr = traffic.get(kernel, {}).get("dram_bytes")
        d = {"kernel": kernel, "units": units, "unit": unit_name, "kernel_ms": k_ms, "e2e_ms": e2e_ms,
             "algorithmic_bytes": int(alg_bytes), "achieved_gbs": ach, "frac_of_hbm_peak": ach / peak_gbs,
             "dram_bytes_ncu": tr, "traffic_over_algorithmic": (tr / alg_bytes) if tr else None,
             "units_per_s_device": units / (k_ms * 1e-3), "cpu_ms_1thread": cpu_ms, "cpu_kind": cpu_kind}
        if extra:
            d.update(extra)
        out[name] = d

    # ---- C2: DepthFilter::updateSeeds, 2000 seeds, 752x480
    c = synth.make_depth_case(2031, 2000, baseline=0.3)
    ref, cur = ctx.frame(c["ref_pyr"]), ctx.frame(c["cur_pyr"])
    dargs = ([ref], [c["T_ref_w"]], cur, c["T_cur_w"], c["cam"], c["ref_index"], c["ftr_px"], c["ftr_f"], c["ftr_level"],
             c["ftr_type"], c["ftr_grad"], c["batch_id"], c["batch_counter"], c["seeds"])
    g = ctx.depth_filter_update(*dargs)
    k_ms, e_ms = timed(lambda: ctx.depth_filter_update(*dargs), 20)
    evals = int(g["n_zmssd"].sum())
    alg = 2000 * (48 + 64 + 400) + 64 * evals + 81 * 10 * int((g["status"] >= 4).sum())
    cpu_ms = None
    if have_ref:
        ob.ref_depth_filter_update([c["ref_pyr"][0]], [c["T_ref_w"]], c["cur_pyr"][0], c["T_cur_w"], 5, c["cam"], c["ref_index"],
                                   c["ftr_px"], c["ftr_f"], c["ftr_level"], c["ftr_type"], c["ftr_grad"], c["batch_id"],
                                   c["batch_counter"], c["seeds"])
        cpu_ms = 1e3 * ob.ref_last_seconds()
    entry("depth_filter_C2", "depth_filter_kernel", 2000, "seeds", alg, k_ms, e_ms, cpu_ms, "reference",
          {"zmssd_evals": evals, "updated": int((g["status"] >= 5).sum())})
    ref.destroy(); cur.destroy()

    # ---- C3: HD 1920x1080, 1000 features: align2D (10 iterations) and pose_optimizer (1000 observations)
    a = synth.make_align_case(3001, 1000, 1920, 1080, n_levels=6)
    fr = ctx.frame(a["pyr"])
    conv, _ = ctx.align2d_batch(fr, a["level"], a["pwb"], a["patch"], 10, a["px_start"])
    k_ms, e_ms = timed(lambda: ctx.align2d_batch(fr, a["level"], a["pwb"], a["patch"], 10, a["px_start"]), 20)
    cpu_ms = None
    if have_ref:
        ob.ref_align2d_batch(a["pyr"][0], 6, a["level"], a["pwb"], a["patch"], 10, a["px_start"])
        cpu_ms = 1e3 * ob.ref_last_seconds()
    entry("align2d_C3", "align_batch_kernel", 1000, "features", 1000 * (100 + 64 + 16 + 81 * 6), k_ms, e_ms, cpu_ms, "reference",
          {"converged": int(conv.sum()), "bytes_note": "81 B x ~6 executed iterations per feature"})
    fr.destroy()
    pc = synth.make_pose_opt_case(1005, 1000, 1920, 1080)
    pargs = (2.0, 10, pc["cam"].fx, pc["T_init"], pc["f"], pc["pos"], pc["level"], pc["has_point"])
    gp = ctx.pose_optimize(*pargs)
    k_ms, e_ms = timed(lambda: ctx.pose_optimize(*pargs), 20)
    cpu_ms = None
    if have_ref:
        ob.ref_pose_optimize(2.0, 10, pc["cam"], pc["T_init"], pc["f"], pc["pos"], pc["level"], pc["has_point"])
        cpu_ms = 1e3 * ob.ref_last_seconds()
    entry("pose_optimizer_C3", "pose_opt_kernel", 1000, "observations", 52 * 1000 * (int(gp["n_iter_done"]) + 2), k_ms, e_ms, cpu_ms,
          "reference", {"iterations": int(gp["n_iter_done"])})
    Bp = 148
    offp = np.arange(Bp + 1, dtype=np.int32) * 1000
    cat = lambda x: np.concatenate([x] * Bp)  # noqa: E731
    bargs = (2.0, 10, [pc["cam"].fx] * Bp, np.stack([pc["T_init"]] * Bp), offp, cat(pc["f"]), cat(pc["pos"]), cat(pc["level"]),
             cat(pc["has_point"]))
    k_ms, e_ms = timed(lambda: ctx.pose_optimize_batch(*bargs), 5)
    entry("pose_optimizer_C3_batch148", "pose_opt_kernel", 1000 * Bp, "observations", Bp * 52 * 1000 * (int(gp["n_iter_done"]) + 2),
          k_ms, e_ms, None, None, {"frames": Bp})

    # ---- Matcher::findMatchDirect, 1000 candidates
    mc = synth.make_match_case(3003, 1000)
    rf, cf = ctx.frame(mc["ref_pyr"]), ctx.frame(mc["cur_pyr"])
    margs = ([rf], [mc["T_ref_w"]], cf, mc["T_cur_w"], mc["cam"], np.zeros(1000, np.int32), mc["ref_px"], mc["ref_f"], mc["ref_level"],
             mc["ftr_type"], mc["ref_grad"], mc["point_pos"], mc["px_cur"], 2)
    k_ms, e_ms = timed(lambda: ctx.find_match_direct(*margs), 20)
    entry("find_match_direct_1000", "find_match_direct_kernel", 1000, "candidates", 1000 * (24 + 68 + 400 + 81 * 6 + 73), k_ms, e_ms,
          None, None)
    rf.destroy(); cf.destroy()

    # ---- row f2: Reprojector::reprojectMap on a 10-keyframe map
    m = synth.make_map_case(4001, n_kfs=10, n_points=1200, n_candidates=150)
    kfs, curf = [ctx.frame(p) for p in m["kf_pyr"]], ctx.frame(m["cur_pyr"])
    rargs = (m["view"], kfs, curf, m["cur_T_f_w"], m["cam"], m["options"], m["cell_order"], m["pt_type"], m["pt_n_failed"],
             m["pt_n_succeeded"])
    gr = ctx.reproject_map(*rargs)
    k_ms, e_ms = timed(lambda: ctx.reproject_map(*rargs), 20)
    cpu_ms = None
    if have_ref:
        ob.ref_reproject_map(m)
        cpu_ms = 1e3 * ob.ref_last_seconds()
    n_spec = int(gr["n_speculative"])
    entry("reprojector_f2", "reproject_match_kernel", n_spec, "aligned points", n_spec * (24 + 16 + 68 + 100 + 81 * 6 + 73), k_ms, e_ms,
          cpu_ms, "reference", {"matches": int(gr["n_matches"]), "trials_sequential": int(gr["n_trials"]),
                                "note": "the CPU aligns only the candidates the cell policy reaches; the GPU aligns every in-frame point"})
    # ---- row f4: FastDetector::detect on a 752x480 keyframe, 3 levels
    det_args = (curf, 30, 3, 20.0)
    gd = ctx.fast_detect(*det_args)
    k_ms, e_ms = timed(lambda: ctx.fast_detect(*det_args), 50)
    cpu_ms = None
    if have_ref:
        ob.ref_fast_detect(m["cur_pyr"][0], 5, 3, 30, 20.0)
        cpu_ms = 1e3 * ob.ref_last_seconds()
    entry("fast_detector_f4", "fast_detect_kernel", int(sum(im.size for im in m["cur_pyr"][:3])), "pixels",
          int(sum(im.size for im in m["cur_pyr"][:3]) + 8 * 26 * 16), k_ms, e_ms, cpu_ms, "reference (over the restated fast library)",
          {"corners": int(gd["n"]), "reference_published_ms": 7.17,
           "reference_published_source": "svo/test/test_feature_detection.cpp:55 (i7-W520, SSE2 fast library)"})
    for fr_ in kfs:
        fr_.destroy()
    curf.destroy()
    # ---- row f3: Point::optimize, 2000 points x 4 observations
    P, n_fr = 2000, 6
    rng = np.random.default_rng(9)
    poses = [synth.se3_mul(synth.se3_exp(np.concatenate([rng.uniform(-0.3, 0.3, 3), rng.uniform(-0.05, 0.05, 3)])), synth.base_pose())
             for _ in range(n_fr)]
    pos = np.stack([rng.uniform(-1, 1, P), rng.uniform(-1, 1, P), rng.uniform(-0.1, 0.1, P)], axis=1)
    obs_fr = np.tile(np.arange(4, dtype=np.int32), P)
    fs = []
    for p_ in range(P):
        for k in range(4):
            v = poses[k][:, :3] @ pos[p_] + poses[k][:, 3]
            fs.append(v / np.linalg.norm(v))
    fs = np.array(fs)
    oargs = (5, pos + rng.normal(0, 0.01, pos.shape), np.arange(P + 1, dtype=np.int32) * 4, obs_fr, fs, poses)
    k_ms, e_ms = timed(lambda: ctx.point_optimize_batch(*oargs), 20)
    entry("point_optimize_f3", "point_optimize_kernel", P, "points", P * (24 + 4 * (24 + 4) * 5 + 24), k_ms, e_ms, None, None)
    # ---- row f1: pyramid build of a 64-frame window (level 0 -> 1 stream kernel + fused levels 2..4)
    imgs = np.random.default_rng(1).integers(0, 256, (64, H, W), dtype=np.uint8)
    pool = capi.FramePool(ctx, W, H, NLEVELS, 64)
    k_ms, e_ms = timed(lambda: (pool.upload(0, 64, imgs.ctypes.data, W * H), ctx.synchronize()), 10)
    entry("pyramid_f1_64_frames", "pyramid_l0_l1_stream_kernel+pyramid_fused_kernel", 64, "frames", 64 * (307200 + 76800 + 76800 + 25200),
          k_ms, e_ms, None, None, {"note": "both pyramid kernels of the upload; e2e includes the pageable 19.7 MB H2D"})
    pool.destroy()
    return out


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
        return

    import torch

    from rpg_svo_b200 import capi, shard

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the CUDA path is the only path (no CPU fallback)")
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    # pin this rank (and the pinned host buffers it is about to allocate) to the NUMA node of its GPU
    props = torch.cuda.get_device_properties(local_rank)
    numa = shard.bind_to_numa_node(shard.numa_node_of_gpu("%04x:%02x:%02x.0" % (props.pci_domain_id, props.pci_bus_id, props.pci_device_id))
                                   if hasattr(props, "pci_bus_id") else None)
    grp = shard.RankGroup("nccl", dev)
    rank, world = grp.rank, grp.world
    B, K, Wm = args.pairs_per_gpu, args.steps, max(args.warmup, 3)
    passes = passes_per_step(K)

    inp = make_inputs(grp.seed, B, f"cuda:{local_rank}")
    ctx = capi.Context(local_rank)
    stream = torch.cuda.ExternalStream(ctx.stream, device=dev)
    host_l0 = inp["level0"].pin_memory()  # [B+1, H, W] uint8, the HOST buffers of the e2e leg
    pool = capi.FramePool(ctx, W, H, NLEVELS, B + 1)  # one slab: one strided H2D copy per window
    frames = pool.frames
    frame_bytes = W * H

    def stage():
        ctx.sia_batch_stage(frames[:B], frames[1:], inp["cam"], inp["T0"], inp["off"], inp["px"], inp["f"],
                            inp["pos"], inp["hp"], inp["ref_pos"], MAX_LEVEL, MIN_LEVEL, NITER)

    def barrier():
        grp.barrier()
        torch.cuda.synchronize()
        ctx.synchronize()

    # ---------------- leg 1: device-resident (value) ----------------
    # clocks / throttle reasons are sampled from here to the end of the e2e leg (both timed regions)
    sampler = ClockSampler(local_rank)
    sampler.start()
    pool.upload(0, B + 1, host_l0.data_ptr(), frame_bytes)
    stage()
    for _ in range(Wm * passes):
        ctx.sia_batch_run()
    barrier()
    l0 = ctx.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(K * passes):
        ctx.sia_batch_run()
    e1.record(stream)
    barrier()
    launches = ctx.launch_count() - l0
    ms_dev_local = e0.elapsed_time(e1)
    value = grp.throughput(B * passes * K, ms_dev_local * 1e-3)
    ms_dev = grp.max_over_ranks(ms_dev_local)
    res = ctx.sia_batch_fetch()
    stats = res["stats"]
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, res)
    alg_bytes = sum(algorithmic_bytes(stats[b], NFEAT) for b in range(B))
    kernel_ms = ms_dev / (K * passes)

    # ---------------- pose RMSE vs the reference's own SparseImgAlign on a sample (not timed) ----------------
    rmse = None
    if rank == 0:
        from oracle import binding as ob  # checker only
        from rpg_svo_b200 import synth

        ob.build()
        n = min(512, B)
        kind, _, run = cpu_runner(ob, synth, inp, n)
        r = run(shard.usable_threads(), want_poses=True)
        if r["T"] is not None:
            err = np.array([synth.pose_error(res["T"][k], r["T"][k]) for k in range(n)])
            gt = np.array([synth.pose_error(res["T"][k], inp["T_gt"][k])[0] for k in range(n)])
            rmse = {"trans_m": float(np.sqrt(np.mean(err[:, 0] ** 2))), "rot_rad": float(np.sqrt(np.mean(err[:, 1] ** 2))),
                    "max_trans_m": float(err[:, 0].max()), "pairs": n, "against": "oracle/_ref (" + kind + ")",
                    "gpu_vs_ground_truth_trans_m": float(np.sqrt(np.mean(gt ** 2)))}

    # ---------------- leg 2: end to end through the C ABI with host buffers ----------------
    e2e = None
    if not args.no_e2e:
        # The window is cut into chunks that alternate between two contexts (= two CUDA streams): while one stream runs the
        # alignment kernel of chunk c, the other copies the images of chunk c+1 over PCIe.  Each chunk owns a private frame
        # pool (pairs k..k+n-1 need frames k..k+n), so nothing is shared between the streams; the boundary frame of a chunk
        # is simply uploaded twice.
        n_chunks = max(1, min(args.e2e_chunks, B))
        ctx2 = capi.Context(local_rank)
        ctxs = [ctx, ctx2]
        bounds = [shard.shard_range(B, c, n_chunks) for c in range(n_chunks)]
        pools = [capi.FramePool(ctxs[c % 2], W, H, NLEVELS, e - b + 1) for c, (b, e) in enumerate(bounds)]
        base = host_l0.data_ptr()
        results = [None] * n_chunks

        def e2e_step():
            for c, (b, e) in enumerate(bounds):
                cx, pl, n = ctxs[c % 2], pools[c], e - b
                fo = inp["off"][b:e + 1] - inp["off"][b]
                sl = slice(b * NFEAT, e * NFEAT)
                if c >= 2:  # the context's staging buffers are about to be reused: drain its previous chunk
                    results[c - 2] = cx.sia_batch_fetch()
                cx.sia_batch_stage(pl.frames[:n], pl.frames[1:n + 1], inp["cam"], inp["T0"][b:e], fo, inp["px"][sl],
                                   inp["f"][sl], inp["pos"][sl], inp["hp"][sl], inp["ref_pos"][b:e], MAX_LEVEL,
                                   MIN_LEVEL, NITER)
                pl.upload(0, n + 1, base + b * frame_bytes, frame_bytes)
                cx.sia_batch_run()
            for c in range(max(0, n_chunks - 2), n_chunks):
                results[c] = ctxs[c % 2].sia_batch_fetch()
            return results

        for _ in range(Wm):
            e2e_step()
        T_chunks = np.concatenate([r["T"] for r in results])
        d = np.array([np.abs(T_chunks[k] - res["T"][k]).max() for k in range(B)])
        assert d.max() < 1e-6, "chunked e2e path disagrees with the device-resident run"
        # a step of this leg = `passes` end-to-end passes over the window, like the device-resident leg
        barrier()
        ctx2.synchronize()
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n_e2e = max(3, min(K * passes, 30))  # bounded: each pass moves ~1.1 GB over PCIe
        s0.record(stream)
        for _ in range(n_e2e):
            e2e_step()  # every fetch synchronises its stream, so all work of the pass is complete here
        s1.record(stream)
        barrier()
        ctx2.synchronize()
        ms_e2e_local = s0.elapsed_time(s1)
        e2e_value = grp.throughput(B * n_e2e, ms_e2e_local * 1e-3)
        for pl in pools:
            pl.destroy()
        ctx2.close()
        h2d = (B + n_chunks) * frame_bytes + B * (272 + ((NFEAT + 15) // 16 * 16) * 65)
        d2h = B * (96 + 288 + 16) + B * NFEAT
        e2e = {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d * passes), "d2h_bytes_per_step": int(d2h * passes),
               "ms_per_pass": grp.max_over_ranks(ms_e2e_local) / n_e2e, "passes_timed": n_e2e,
               "h2d_bytes_per_pass": int(h2d), "d2h_bytes_per_pass": int(d2h)}

    clocks = sampler.stop()
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    else:
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"

    extras = {}
    if rank == 0 and not args.no_extras:
        extras = measure_latency_and_c4(ctx, capi, torch, stream, inp, host_l0, pool)
        if world == 1:
            extras["roofline_by_kernel"] = measure_kernels(ctx, capi, peak)

    # ---------------- CPU baseline (rank 0, N == 1 only) ----------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        from oracle import binding as ob
        from rpg_svo_b200 import synth

        n = min(args.cpu_sample, B)
        kind, note, run = cpu_runner(ob, synth, inp, n)
        run(1)
        reps, dt = 0, 0.0
        while dt < 10.0 and reps < 40:
            dt += run(1)["seconds"]
            reps += 1
        cpu = {"value": n * reps / dt, "unit": UNIT, "cores": 1, "kind": kind,
               "sample": f"first {n} frame pairs of the step x {reps} passes, single thread", "host": shard.host_cpu_limits(),
               "note": note}

    if rank == 0:
        achieved = alg_bytes / (kernel_ms * 1e-3) / 1e9
        traffic = None
        prof = os.path.join(ROOT, "profiles", "sia_kernel_dram.json")
        if os.path.exists(prof):
            pj = json.load(open(prof))
            if pj.get("pairs_per_launch") == B:
                traffic = pj.get("dram_bytes_per_launch")
        cfg = make_config(args)
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": Wm,
                "ms_per_step": ms_dev / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32 interpolation/residuals + f64 geometry/normal equations (as the reference)",
                "data": "synthetic", "config": cfg,
                "pose_rmse_vs_ref": rmse,
                "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                             "traffic": traffic, "peak_source": peak_src, "kernel": "svo::sia_kernel<FPT=2,EVAL=false,MAXT=160,MINB=3,CS=1,CG=false,UP=false>",
                             "algorithmic_bytes_per_launch": alg_bytes, "kernel_ms": kernel_ms,
                             "mean_gn_iterations_per_pair": float(np.mean(stats["n_iters"])),
                             "note": "latency-bound sparse gather kernel (ncu r02h: see profiles/ and DESIGN.md 4.1 for the stall breakdown and the sector-granular DRAM floor)"},
                "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks, "numa": numa}
        line.update(extras)
        print(json.dumps(line), flush=True)
    grp.close()
    pool.destroy()
    ctx.close()


if __name__ == "__main__":
    main()
