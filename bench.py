#!/usr/bin/env python
"""bench.py -- headline benchmark of the hot path (BASELINE.json: "1920x1080i YV12 frames/sec (logo-eval + combing)").

    python bench.py [--gpus N] [--steps K] [--warmup W]            # this repo's CUDA path (torchrun for N > 1)
    python bench.py --impl reference [--gpus N] [--steps K] ...    # the reference's CPU path on the host cores
    python bench.py --config {comb_1440,logoscan_10k,logo_analyze,logo_scan}   # secondary BASELINE configs, one JSON line
    python bench.py --dump-outputs DIR ...                        # + the last timed step's results as DIR/{scores,counts}.npy

One step = one pass of the fused hot path (LogoFrame::ScanFrame logo evaluation, 1 logo, fades {0,1}, + the
combing / field-difference counters) over ONE synthetic 1800-frame 1920x1080i YV12 clip (BASELINE.json configs[1]),
resident in HBM (5.6 GB >> 126 MB L2, so no L2 flush is needed between steps).  N GPUs = N independent clips, one per
rank (weak scaling), with ONE NCCL all-gather of the per-frame results per step, issued on a side stream.
Prints ONE JSON line on rank 0.  The line carries a `parity` block: the WHOLE clip's GPU results compared with the
reference's own code (logo scores, bitwise) and the combing spec (counters) -- a mismatch exits non-zero.
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

W, H = 1920, 1080
CLIP_FRAMES = 1800
FRAME_BYTES = W * H * 3 // 2
IMGX, IMGY, LOGO_W, LOGO_H = 1700, 60, 64, 64
MASKRATIO = 0.35
SEED = 0x5EED0001
METRIC = "1920x1080i YV12 frames/sec (logo-eval + combing)"
WORKLOAD = "1920x1080i 1800-frame synthetic clip, AMTLogo eval every frame + combing (configs[1])"
COMB_NOTE = ("combing half = this repo's spec in AVX2 (oracle/amtk_comb_avx2.c) -- NOT Amatsukaze code: the reference "
             "has no implementation of it (external KFM plugin)")


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (measured copy bandwidth)"
    except Exception:
        return 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md; MEASURED_PEAKS.json absent)"


def staged_h2d_bytes(nframes, frame_bytes, budget=256 << 20):
    """Bytes the library copies host->device for one pass over a host clip: chunks of the staging budget, each chunk
    after the first re-sends one halo frame for the inter-frame difference (for_each_window in csrc/amtk_b200.cu)."""
    per = max(1, min(nframes, budget // frame_bytes))
    if per > 1:
        per -= 1
    chunks = (nframes + per - 1) // per
    return (nframes + chunks - 1) * frame_bytes


def bind_to_gpu_numa(index):
    """Pin this process to the CPUs next to GPU `index` (NVML's ideal affinity) BEFORE any pinned host allocation, so
    the staging memory of the end-to-end path sits on the GPU's own NUMA node (8-GPU e2e scaled 0.675 without it)."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        before = len(os.sched_getaffinity(0))
        pynvml.nvmlDeviceSetCpuAffinity(h)
        after = sorted(os.sched_getaffinity(0))
        return {"cpus": len(after), "cpus_before": before, "first": after[0], "last": after[-1]}
    except Exception as e:      # no NVML / not permitted: run unbound
        return {"error": str(e)[:80]}


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons of one GPU through NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self.active = False
        self.stop_flag = False
        self.ok = True
        try:
            import pynvml
            self.nv = pynvml
            pynvml.nvmlInit()
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {}
        for nm in ("HwSlowdown", "HwThermalSlowdown", "SwThermalSlowdown", "SwPowerCap", "HwPowerBrakeSlowdown"):
            for prefix in ("nvmlClocksEventReason", "nvmlClocksThrottleReason"):
                v = getattr(nv, prefix + nm, None)
                if v is not None:
                    names[v] = nm
                    break
        while not self.stop_flag:
            try:
                mhz = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                if self.active:
                    self.samples.append(mhz)
                    for bit, nm in names.items():
                        if r & bit:
                            self.reasons.add(nm)
            except Exception:
                pass
            time.sleep(0.005)

    def summary(self):
        if not self.ok or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0}
        s = sorted(self.samples)
        snake = {"HwSlowdown": "hw_slowdown", "HwThermalSlowdown": "hw_thermal_slowdown",
                 "SwThermalSlowdown": "sw_thermal_slowdown", "SwPowerCap": "sw_power_cap",
                 "HwPowerBrakeSlowdown": "hw_power_brake_slowdown"}
        return {"sm_mhz": s[len(s) // 2], "sm_max_mhz": self.max_mhz, "reasons": sorted(snake[r] for r in self.reasons),
                "samples": len(s)}


def dump_outputs(d, scores, counts):
    """--dump-outputs: what the timed path handed its caller in the last timed step, in one layout for every arm, one row per
    clip (= per GPU): DIR/scores.npy float32 (clips, frames, 2) and DIR/counts.npy (clips, frames, 12), the int32 counters
    widened to float64 (exact).  The inputs are seeded, so two builds run with the same arguments can be compared output
    for output."""
    import numpy as np
    os.makedirs(d, exist_ok=True)
    np.save(os.path.join(d, "scores.npy"), np.asarray(scores, np.float32).reshape(-1, CLIP_FRAMES, 2))
    np.save(os.path.join(d, "counts.npy"), np.asarray(counts).astype(np.float64).reshape(-1, CLIP_FRAMES, 12))


def make_clip(torch, synth, logo, device, seed, w=W, h=H, nframes=CLIP_FRAMES, mode="interlaced", imgx=IMGX, imgy=IMGY, out=None):
    """A synthetic clip generated on the GPU in chunks (integer-only generator, identical on CPU and CUDA)."""
    fb = w * h * 3 // 2
    clip = torch.empty((nframes, fb), dtype=torch.uint8, device=device) if out is None else out
    step = 20
    for n0 in range(0, nframes, step):
        n = min(step, nframes - n0)
        synth.make_frames(n0, n, w, h, seed=seed, device=device, mode=mode, logo=logo, imgx=imgx, imgy=imgy, out=clip[n0:n0 + n])
    return clip


# ---------------------------------------------------------------------------------------------------------------
# CPU arm
# ---------------------------------------------------------------------------------------------------------------
def cpu_measure(po, frames, logo_data, th6, threads, passes=3, one_thread_frames=48):
    """Times the CPU implementation on `frames` (numpy (n, FRAME_BYTES)): all usable threads (best of `passes`, plus the
    logo-only and comb-only splits) and ONE thread -- how the reference really runs this path -- on a short prefix.
    Returns (dict for cpu_baseline, scores, counts) with the results of the all-thread fused pass."""
    n = frames.shape[0]
    bN = po.CpuBench(W, H, logo_data, IMGX, IMGY, threads, MASKRATIO)
    best, sc, cn = None, None, None
    for _ in range(passes):
        sec, sc, cn = bN.run(frames, th6, 3, "avx2")
        best = sec if best is None else min(best, sec)
    logo_sec = min(bN.run(frames, th6, 1, "avx2")[0] for _ in range(2))
    comb_sec = min(bN.run(frames, th6, 2, "avx2")[0] for _ in range(2))
    scal_n = min(n, max(threads, 16))
    scal_sec = bN.run(frames[:scal_n], th6, 2, "scalar")[0]
    kind = bN.kind
    bN.close()
    b1 = po.CpuBench(W, H, logo_data, IMGX, IMGY, 1, MASKRATIO)
    n1 = min(n, one_thread_frames)
    one = min(b1.run(frames[:n1], th6, 3, "avx2")[0] for _ in range(2))
    one_logo = min(b1.run(frames[:n1], th6, 1, "avx2")[0] for _ in range(2))
    b1.close()
    info = {"value": n / best, "unit": "frames/s", "cores": threads, "threads": threads, "kind": kind,
            "threads_N": n / best, "threads_1": n1 / one,
            "logo_only": {"threads_N": n / logo_sec, "threads_1": n1 / one_logo, "code": "reference's own ComputeKernel.cpp/LogoScan.hpp (oracle/_ref)" if kind == "reference" else "C port (oracle/amtk_oracle.c)"},
            "comb_only": {"threads_N": n / comb_sec, "threads_N_scalar_spec": scal_n / scal_sec, "code": "this repo's spec, AVX2 (not Amatsukaze code)"},
            "host_cpus_online": os.cpu_count(),
            "sample": "%d frames per pass (%.1f per thread), best of %d passes, thread team and scratch created outside the timed "
                      "region; threads = affinity mask capped by the cgroup quota; logo half = %s; %s; 1-thread figure on %d frames"
                      % (n, n / threads, passes, "reference's own code (oracle/_ref)" if kind == "reference" else "C port", COMB_NOTE, n1)}
    return info, sc, cn


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU code (oracle/_ref) for the logo half + this repo's AVX2 comb spec for the
    combing half (absent from the reference), on all usable host threads, on a bounded sample of the same workload."""
    if rank != 0:
        return
    import numpy as np
    import torch
    from amatsukaze_b200 import synth
    from oracle import pyoracle as po
    threads = po.usable_cpu_threads()
    sample = args.ref_frames if args.ref_frames > 0 else max(96, min(CLIP_FRAMES, 8 * threads))
    logo = synth.make_logo(LOGO_W, LOGO_H)
    gen = "cpu"
    if torch.cuda.is_available() and sample > 64:       # input generation only; the measured code runs on the host cores
        gen = "cuda (input generation only)"
        frames = make_clip(torch, synth, logo, "cuda", SEED, nframes=sample).cpu().numpy()
    else:
        uniq = min(sample, 64)                           # CPU generation is slow: tile a 64-frame unique set
        base = np.concatenate([synth.make_frames(CLIP_FRAMES // 3 + i, min(8, uniq - i), W, H, seed=SEED, logo=logo,
                                                 imgx=IMGX, imgy=IMGY).numpy() for i in range(0, uniq, 8)])
        frames = np.concatenate([base] * ((sample + uniq - 1) // uniq))[:sample]
    th = [20, 12, 36, 24, 16, 48]
    b = po.CpuBench(W, H, logo["data"], IMGX, IMGY, threads, MASKRATIO)
    for _ in range(args.warmup):
        b.run(frames, th, 3, "avx2")
    total, best = 0.0, None
    for _ in range(args.steps):
        sec = b.run(frames, th, 3, "avx2")[0]
        total += sec
        best = sec if best is None else min(best, sec)
    kind = b.kind
    b.close()
    b1 = po.CpuBench(W, H, logo["data"], IMGX, IMGY, 1, MASKRATIO)
    n1 = min(sample, 48)
    one = min(b1.run(frames[:n1], th, 3, "avx2")[0] for _ in range(2))
    b1.close()
    fps = sample * args.steps / total
    line = {
        "impl": "reference", "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u8+f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "frames_per_step": sample, "logo": "64x64 @(1700,60) maskratio 0.35, fades {0,1}",
                   "input_generated_on": gen},
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": threads, "threads": threads, "kind": kind,
                         "threads_N": fps, "threads_N_best_step": sample / best, "threads_1": n1 / one,
                         "host_cpus_online": os.cpu_count(),
                         "sample": "%d frames per step (%.1f per thread); threads = affinity mask capped by the cgroup quota; thread "
                                   "team and scratch created outside the timed region; logo half = %s; %s"
                                   % (sample, sample / threads,
                                      "reference's own ComputeKernel.cpp/LogoScan.hpp code (oracle/_ref)" if kind == "reference" else "C port (oracle/amtk_oracle.c)",
                                      COMB_NOTE)},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------------------
# secondary BASELINE configs (device-resident, CUDA events on the context's stream)
# ---------------------------------------------------------------------------------------------------------------
def timed_ms(torch, stream, fn, reps):
    fn()
    stream.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(reps):
        fn()
    e1.record(stream)
    stream.synchronize()
    return e0.elapsed_time(e1) / reps


def secondary_configs(torch, ab, synth, ctx, stream, device, which, peak, po=None):
    """configs[0] (one 1440x1080 frame, 64x64 template: call latency), configs[2] (1440x1080 3600-field combing pass),
    configs[3] (LogoScan accumulation over 10000 1080p frames), AMTAnalyzeLogo (33 evaluations per frame) and
    LogoFrame::ScanFrame alone, each device resident.  `po` (the oracle module) is passed only by the cpu_baseline leg."""
    import numpy as np
    out = {}
    lg = synth.make_logo(LOGO_W, LOGO_H)
    with torch.cuda.stream(stream):
        if "single_frame_1440" in which:
            # configs[0]: ONE 1440x1080 YV12 frame, 64x64 template at (1280, 64), DeintY + EvaluateLogo(fade 0) + EvaluateLogo(fade 1)
            # (SURVEY 8(d) config 1).  This is a latency case: one GetFrame-sized call through the C ABI.
            w, h, ix, iy = 1440, 1080, 1280, 64
            t = make_clip(torch, synth, lg, device, SEED + 3, w, h, 1, imgx=ix, imgy=iy)
            logo1 = ab.Logo.create(lg["data"], LOGO_W, LOGO_H, w, h, ix, iy).deint().create_mask(MASKRATIO)
            hfr = torch.empty((1, w * h * 3 // 2), dtype=torch.uint8, pin_memory=True)
            hfr.copy_(t)
            torch.cuda.synchronize()
            dclip, hclip = ab.yv12_clip(t, w, h, 1, True), ab.yv12_clip(hfr, w, h, 1, on_device=False)
            hs, hd = np.empty((1, 1, 2), np.float32), np.empty((1, 1, 2), np.float32)
            reps = 300
            for clip1, dst, key in ((hclip, hs, "host_frame_us_per_call"), (dclip, hd, "resident_frame_us_per_call")):
                for _ in range(20):
                    ctx.scan_frames(clip1, [logo1], out=dst)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                for _ in range(reps):
                    ctx.scan_frames(clip1, [logo1], out=dst)        # blocking: returns after the D2H of the two scores
                out.setdefault("single_frame_1440", {})[key] = (time.perf_counter() - t0) / reps * 1e6
            e = out["single_frame_1440"]
            e["workload"] = "configs[0]: one 1440x1080 YV12 frame, 64x64 template at (1280,64), ScanFrame (2 evaluations), wall clock per blocking C-ABI call"
            e["h2d_bytes_per_call_host_frame"] = ctx.last_h2d_bytes if hasattr(ctx, "last_h2d_bytes") else None
            e["host_equals_resident"] = bool(np.array_equal(hs.view(np.uint32), hd.view(np.uint32)))
            if po is not None:
                b1 = po.CpuBench(w, h, lg["data"], ix, iy, 1, MASKRATIO)
                fr = np.repeat(hfr.numpy(), 64, axis=0)
                sec, sc, _ = min((b1.run(fr, [20, 12, 36, 24, 16, 48], 1, "avx2") for _ in range(3)), key=lambda r: r[0])
                e["cpu_us_per_frame_1_thread"] = sec / 64 * 1e6
                e["cpu_code"] = "reference's own ComputeKernel.cpp/LogoScan.hpp (oracle/_ref)" if b1.kind == "reference" else "C port (oracle/amtk_oracle.c)"
                e["scores_bitexact_vs_cpu"] = bool(np.array_equal(sc[:1].view(np.uint32), hd.reshape(1, 2).view(np.uint32)))
                b1.close()
            del t, hfr
            # AMTAnalyzeLogo::GetFrame (LogoScan.hpp:1119-1161): ONE output frame = 8 source frames x 33 evaluations
            # (deint logo + two field logos x 11 fades), the call AviSynth makes; 8 host frames in, 1056 bytes out
            t8 = make_clip(torch, synth, lg, device, SEED + 5, w, h, 8, imgx=ix, imgy=iy)
            raw = ab.Logo.create(lg["data"], LOGO_W, LOGO_H, w, h, ix, iy)
            de, top, bot = raw.deint().create_mask(MASKRATIO), raw.field(0).create_mask(MASKRATIO), raw.field(1).create_mask(MASKRATIO)
            h8 = torch.empty((8, w * h * 3 // 2), dtype=torch.uint8, pin_memory=True)
            h8.copy_(t8)
            torch.cuda.synchronize()
            hclip8 = ab.yv12_clip(h8, w, h, 8, on_device=False)
            ha = np.empty((8, 33), np.float32)
            for _ in range(10):
                ctx.analyze_frames(hclip8, de, top, bot, out=ha)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(100):
                ctx.analyze_frames(hclip8, de, top, bot, out=ha)
            g = {"workload": "AMTAnalyzeLogo::GetFrame: one output frame = 8 host source frames (1440x1080) x 33 evaluations, wall clock per blocking C-ABI call",
                 "us_per_call": (time.perf_counter() - t0) / 100 * 1e6, "h2d_bytes_per_call": ctx.last_h2d_bytes, "d2h_bytes_per_call": int(ha.nbytes)}
            if po is not None and po.ref_available():
                rl = po.RefLogo.create(lg["data"], LOGO_W, LOGO_H, w, h, ix, iy)
                rde, rtop, rbot = rl.deint().create_mask(MASKRATIO), rl.field(0).create_mask(MASKRATIO), rl.field(1).create_mask(MASKRATIO)
                Y8 = h8.numpy()[:, : w * h].reshape(8, h, w)
                best, ra = None, None
                for _ in range(2):
                    t0 = time.perf_counter()
                    ra = np.stack([po.ref_analyze_frame(rde, rtop, rbot, Y8[i]) for i in range(8)])
                    dt = time.perf_counter() - t0
                    best = dt if best is None else min(best, dt)
                g["cpu_us_per_call_1_thread"] = best * 1e6
                g["cpu_code"] = "reference's own DeintY/CopyY/EvaluateLogo (oracle/_ref), 33 x 8 calls through ctypes (a few % of binding overhead)"
                g["bitexact_vs_cpu"] = bool(np.array_equal(ra.view(np.uint32), ha.view(np.uint32)))
            out["analyze_getframe_1440"] = g
            # AMTEraseLogo::GetFrame (LogoScan.hpp:1343-1397): Delogo on the Y, U, V rectangles of ONE host frame, in place
            # (per-field fades: the two-pass form); only the three rectangles cross PCIe, both ways
            h1 = h8[:1].clone().pin_memory()
            orig = h1.numpy().copy()
            hclip1 = ab.yv12_clip(h1, w, h, 1, on_device=False)
            fd = np.array([[0.3, 0.9]], np.float32)
            for _ in range(10):
                h1.numpy()[:] = orig
                ctx.erase_logo(hclip1, raw, fd)
            erased = h1.numpy().copy()
            t0 = time.perf_counter()
            for _ in range(100):
                ctx.erase_logo(hclip1, raw, fd)                    # (erases the erased frame again: same work, timing only)
            ge = {"workload": "AMTEraseLogo::GetFrame: Delogo of the 64x64 Y and 32x32 U, V rectangles of one 1440x1080 host frame, in place, per-field fades, wall clock per blocking C-ABI call",
                  "us_per_call": (time.perf_counter() - t0) / 100 * 1e6, "h2d_bytes_per_call": ctx.last_h2d_bytes}
            if po is not None:
                ol = po.OracleLogo.create(lg["data"], LOGO_W, LOGO_H, w, h, ix, iy)
                best, ref_fr = None, None
                for _ in range(5):
                    t0 = time.perf_counter()
                    ref_fr = orig.copy()                           # the reference's MakeWritable: a full-frame copy (:1347)
                    Yp, Up, Vp = (ref_fr[0, : w * h].reshape(h, w), ref_fr[0, w * h: w * h * 5 // 4].reshape(h // 2, w // 2),
                                  ref_fr[0, w * h * 5 // 4:].reshape(h // 2, w // 2))
                    po.or_erase_frame(ol, Yp, Up, Vp, 0.3, 0.9)
                    dt = time.perf_counter() - t0
                    best = dt if best is None else min(best, dt)
                ge["cpu_us_per_frame_1_thread"] = best * 1e6
                ge["cpu_code"] = "C port of Delogo/GetFrameT (oracle/amtk_oracle.c) + the full-frame MakeWritable copy the reference makes"
                ge["bytes_equal_vs_cpu"] = bool(np.array_equal(erased, ref_fr))
            out["erase_getframe_1440"] = ge
            del t8, h8, h1
        if "comb_1440" in which:
            w, h, n = 1440, 1080, 1800
            t = make_clip(torch, synth, None, device, SEED, w, h, n, mode="telecine")
            clip = ab.yv12_clip(t, w, h, n, True)
            res = torch.empty((n, 12), dtype=torch.int32, device=device)
            ms = timed_ms(torch, stream, lambda: ctx.comb_frames(clip, out=res), 20)
            gbs = n * w * h * 1.5 / ms / 1e6
            out["comb_1440"] = {"workload": "configs[2]: 1440x1080i 3600-field KFM combing/field-diff pass, 1800 frames resident",
                                "ms": ms, "frames_per_s": n / ms * 1e3, "fields_per_s": 2 * n / ms * 1e3,
                                "algorithmic_gbs": gbs, "frac_of_measured_hbm": gbs / peak}
            del t, clip
        if "comb_p10" in which:
            # YUV420P10 (north_star: "YV12/YUV420P10 planes"): 16-bit containers, 10 significant bits, 900 frames = 5.6 GB resident
            w, h, n = 1920, 1080, 900
            t8 = make_clip(torch, synth, None, device, SEED, w, h, n, mode="telecine")
            t = torch.empty((n, w * h * 3 // 2), dtype=torch.int16, device=device)
            for k in range(0, n, 50):
                v = t8[k:k + 50].to(torch.int32)
                t[k:k + 50] = (v * 4 + (v & 3)).to(torch.int16)
            del t8
            clip = ab.yv12_clip(t, w, h, n, True, bits=10)
            p10 = ab.default_comb_params()
            p10.th_move_y, p10.th_shima_y, p10.th_lshima_y = 80, 48, 144
            p10.th_move_c, p10.th_shima_c, p10.th_lshima_c = 96, 64, 192
            res = torch.empty((n, 12), dtype=torch.int32, device=device)
            ms = timed_ms(torch, stream, lambda: ctx.comb_frames(clip, p10, out=res), 20)
            gbs = n * w * h * 3.0 / ms / 1e6
            out["comb_p10"] = {"workload": "1920x1080i YUV420P10 combing/field-diff pass, 900 frames (5.6 GB) resident",
                               "ms": ms, "frames_per_s": n / ms * 1e3, "algorithmic_gbs": gbs, "frac_of_measured_hbm": gbs / peak}
            del t, clip
        if "logoscan_10k" in which:
            w, h, n = 1920, 1080, 10000
            t = make_clip(torch, synth, lg, device, SEED + 7, w, h, n, mode="flat")
            clip = ab.yv12_clip(t, w, h, n, True)
            for (sw, sh) in ((64, 64), (256, 128)):
                acc = ctx.logo_scan(sw, sh, 12)
                sx = IMGX if sw == 64 else 1600
                ms = timed_ms(torch, stream, lambda: acc.add_frames(clip, sx, IMGY), 3)
                out["logoscan_10k_%dx%d" % (sw, sh)] = {
                    "workload": "configs[3]: LogoScan::AddFrame over 10000 resident 1920x1080 frames, ROI %dx%d, thy 12" % (sw, sh),
                    "ms": ms, "frames_per_s": n / ms * 1e3, "roi_gbs": n * sw * sh * 1.5 / ms / 1e6,
                    "note": "host-pointer validity output (10 kB D2H + sync) is inside the timing"}
                del acc
            del t, clip
        if "logo_analyze" in which or "logo_scan" in which:
            n = CLIP_FRAMES
            t = make_clip(torch, synth, lg, device, SEED)
            clip = ab.yv12_clip(t, W, H, n, True)
            raw = ab.Logo.create(lg["data"], LOGO_W, LOGO_H, W, H, IMGX, IMGY)
            de, top, bot = raw.deint().create_mask(MASKRATIO), raw.field(0).create_mask(MASKRATIO), raw.field(1).create_mask(MASKRATIO)
            if "logo_scan" in which:
                res = torch.empty((n, 1, 2), dtype=torch.float32, device=device)
                ms = timed_ms(torch, stream, lambda: ctx.scan_frames(clip, [de], out=res), 20)
                out["logo_scan"] = {"workload": "LogoFrame::ScanFrame alone (2 evaluations/frame), 1800 resident 1080p frames",
                                    "ms": ms, "frames_per_s": n / ms * 1e3}
            if "logo_analyze" in which:
                res = torch.empty((n, 33), dtype=torch.float32, device=device)
                ms = timed_ms(torch, stream, lambda: ctx.analyze_frames(clip, de, top, bot, out=res), 5)
                out["logo_analyze"] = {"workload": "AMTAnalyzeLogo (33 evaluations/frame: deint + 2 field logos x 11 fades), 1800 resident 1080p frames",
                                       "ms": ms, "frames_per_s": n / ms * 1e3, "evals_per_s": 33 * n / ms * 1e3}
            del t, clip
    torch.cuda.empty_cache()
    return out


# ---------------------------------------------------------------------------------------------------------------
# this repo's arm
# ---------------------------------------------------------------------------------------------------------------
def run_group(args):
    """python bench.py --gpus N WITHOUT torchrun: one process drives N GPUs through the library's group API
    (amtk_group_create: a context, a stream and a host thread per device, each thread bound to its GPU's CPUs;
    ncclCommInitAll; one ncclAllGather of the per-frame results per pass).  Same workload, metric and JSON line as the
    torchrun arm; timed on the devices (one CUDA event pair per GPU, maximum taken)."""
    import numpy as np
    import torch
    import amatsukaze_b200 as ab
    from amatsukaze_b200 import synth
    assert torch.cuda.is_available() and torch.cuda.device_count() >= args.gpus, "bench.py needs %d B200s" % args.gpus
    n = args.gpus
    g = ab.Group(n)
    logo_def = synth.make_logo(LOGO_W, LOGO_H)
    prm = ab.default_comb_params()
    tensors, clips, logos = [], [], []
    for i in range(n):
        t = make_clip(torch, synth, logo_def, torch.device("cuda", i), SEED + i)
        tensors.append(t)
        clips.append(ab.yv12_clip(t, W, H, CLIP_FRAMES, on_device=True))
        logos.append(ab.Logo.create(logo_def["data"], LOGO_W, LOGO_H, W, H, IMGX, IMGY).deint().create_mask(MASKRATIO))
    torch.cuda.synchronize()
    sampler = ClockSampler(0)
    sampler.start()
    for _ in range(max(args.warmup, 3)):
        g.scan_comb_streams(clips, logos, prm, CLIP_FRAMES)
    g.synchronize()
    c0 = g.ctx(0)
    l0 = c0.launches
    c0.kernel_timing(reset=True)
    c0.set_kernel_timing(True)
    sampler.active = True
    g.mark(0)
    for _ in range(args.steps):
        g.scan_comb_streams(clips, logos, prm, CLIP_FRAMES)
    g.mark(1)
    g.synchronize()
    sampler.active = False
    per_dev = g.elapsed_ms(0, 1)
    elapsed_ms = max(per_dev)
    comb_ms, comb_n = c0.kernel_timing(reset=True)
    c0.set_kernel_timing(False)
    launches = (c0.launches - l0) * n
    value = CLIP_FRAMES * n * args.steps / (elapsed_ms * 1e-3)
    d_scores, d_counts = g.fetch_results(CLIP_FRAMES, 0)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, d_scores, d_counts)
    # ---- end to end: pinned, NUMA-local host clips, one per GPU, staged concurrently by the members' own threads ----
    e2e = None
    hosts = []
    if not args.no_e2e:
        for i in range(n):
            hb = g.host_alloc(i, CLIP_FRAMES * FRAME_BYTES).reshape(CLIP_FRAMES, FRAME_BYTES)
            hb[:] = tensors[i].cpu().numpy()
            hosts.append(hb)
        hclips = [ab.yv12_clip(hb, W, H, CLIP_FRAMES, on_device=False) for hb in hosts]
        g.scan_comb_streams(hclips, logos, prm, CLIP_FRAMES)             # warm-up (staging buffers)
        g.synchronize()
        g.mark(2)
        for _ in range(args.e2e_steps):
            g.scan_comb_streams(hclips, logos, prm, CLIP_FRAMES)
            h_scores, h_counts = g.fetch_results(CLIP_FRAMES, 0)           # D2H of the gathered results, every step
        g.mark(3)
        g.synchronize()
        e2e_ms = max(g.elapsed_ms(2, 3))
        same = bool(np.array_equal(h_scores, d_scores) and np.array_equal(h_counts, d_counts))
        h2d = staged_h2d_bytes(CLIP_FRAMES, FRAME_BYTES)
        e2e = {"value": CLIP_FRAMES * n * args.e2e_steps / (e2e_ms * 1e-3), "unit": "frames/s", "h2d_bytes_per_step": h2d * n,
               "d2h_bytes_per_step": int(h_scores.nbytes + h_counts.nbytes), "steps": args.e2e_steps,
               "host_memory": "pinned, allocated by each member's CPU-bound thread (NUMA-local)",
               "numa_cpus_per_member": [g.numa_cpus(i) for i in range(n)], "matches_device_run": same,
               "h2d_gbs_per_gpu": h2d * args.e2e_steps / (e2e_ms * 1e-3) / 1e9,
               "note": "PCIe-bound by construction: every frame byte crosses the host link once"}
    read_ceiling = c0.probe_read_gbs(tensors[0], reps=3)
    sampler.stop_flag = True
    peak, peak_src = measured_peak_gbs()
    alg_bytes = CLIP_FRAMES * FRAME_BYTES
    avg_ms = comb_ms / max(comb_n, 1)
    achieved = alg_bytes / (avg_ms * 1e-3) / 1e9
    cpu, parity, exit_code = None, None, 0
    if not args.no_cpu:
        from oracle import pyoracle as po
        threads = po.usable_cpu_threads()
        fr = hosts[0] if hosts else tensors[0].cpu().numpy()
        cpu, sc, cn = cpu_measure(po, np.ascontiguousarray(fr), logo_def["data"], prm.as_list(), threads)
        s_ok = bool(np.array_equal(d_scores[0].view(np.uint32), sc.view(np.uint32)))
        c_ok = bool(np.array_equal(d_counts[0], cn))
        parity = {"frames": CLIP_FRAMES, "scores_bitexact": s_ok, "counts_equal": c_ok, "oracle": cpu["kind"],
                  "checked": "member 0's clip, whole clip, through the gathered result block"}
        if not (s_ok and c_ok):
            exit_code = 3
    line = {
        "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": n, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": elapsed_ms / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u8+f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "frames_per_step_per_gpu": CLIP_FRAMES, "logo": "64x64 @(1700,60) maskratio 0.35, fades {0,1}",
                   "l2": "step input 5.6 GB per GPU is larger than the 126 MB L2 (no flush needed)",
                   "parallelism": "single process, amtk_group: one independent clip per GPU, host thread + stream per device, "
                                  "one ncclAllGather of the results per step on a side stream (NCCL %d)" % g.nccl_version},
        "ms_per_step_per_gpu": [m / args.steps for m in per_dev],
        "clocks": sampler.summary(), "e2e": e2e, "gpu_launches": int(launches),
        "roofline": {"bound": "hbm", "kernel": "comb_ws_kernel (8-bit streaming pass, member 0)", "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak, "traffic": None, "peak_source": peak_src, "algorithmic_bytes_per_launch": alg_bytes,
                     "avg_launch_ms": avg_ms, "launches_timed": int(comb_n), "share_of_step": comb_ms / max(elapsed_ms, 1e-9),
                     "read_only_ceiling_gbs": read_ceiling},
        "cpu_baseline": cpu, "parity": parity,
    }
    print(json.dumps(line), flush=True)
    g.close()
    if exit_code:
        sys.stderr.write("bench.py: PARITY MISMATCH against the CPU oracle (see the `parity` block)\n")
        sys.exit(exit_code)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="headline",
                    choices=["headline", "single_frame_1440", "comb_1440", "comb_p10", "logoscan_10k", "logo_analyze", "logo_scan", "secondary"])
    ap.add_argument("--ref-frames", type=int, default=0, help="frames per step of the CPU reference arm (0 = 8 per thread, 96..1800)")
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true", help="skip the CPU baseline AND the full-clip parity check")
    ap.add_argument("--no-secondary", action="store_true", help="skip the secondary configs in the headline line")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the results of the last timed step of the headline run (per-frame logo scores and combing "
                         "counters) as DIR/scores.npy and DIR/counts.npy; not with --impl reference or --config")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "b200" or args.config != "headline"):
        ap.error("--dump-outputs writes the results of the headline run of this repo's CUDA path: "
                 "it cannot be combined with --impl reference or --config")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world == 1 and args.gpus > 1:
        run_group(args)         # ONE process, the library's own multi-GPU driver (amtk_group_*: thread + stream per device, NCCL gather)
        return

    import numpy as np
    import torch
    import torch.distributed as dist
    import amatsukaze_b200 as ab
    from amatsukaze_b200 import synth

    assert torch.cuda.is_available(), "bench.py needs a B200 (no CPU fallback)"
    numa = bind_to_gpu_numa(local_rank) if world > 1 else {"unbound": "single GPU run"}
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)

    stream = torch.cuda.Stream(device=device)
    ctx = ab.Context(local_rank, stream.cuda_stream)
    peak, peak_src = measured_peak_gbs()

    if args.config != "headline":
        which = ["single_frame_1440", "comb_1440", "comb_p10", "logoscan_10k", "logo_analyze", "logo_scan"] if args.config == "secondary" else [args.config]
        po = None
        if not args.no_cpu and "single_frame_1440" in which:     # the CPU figures beside the GetFrame-sized calls (cpu_baseline leg)
            from oracle import pyoracle as po
        res = secondary_configs(torch, ab, synth, ctx, stream, device, which, peak, po=po)
        if rank == 0:
            print(json.dumps({"config": args.config, "n_gpus": 1, "data": "synthetic", "timing": "CUDA events on the launch stream, device-resident inputs",
                              "peak_gbs": peak, "results": res}), flush=True)
        ctx.close()
        return

    logo_def = synth.make_logo(LOGO_W, LOGO_H)
    logo = ab.Logo.create(logo_def["data"], LOGO_W, LOGO_H, W, H, IMGX, IMGY).deint().create_mask(MASKRATIO)
    prm = ab.default_comb_params()

    clip_t = make_clip(torch, synth, logo_def, device, SEED + rank)
    torch.cuda.synchronize()
    clip = ab.yv12_clip(clip_t, W, H, CLIP_FRAMES, on_device=True)
    # per-frame results of one pass live back to back in ONE buffer so that the final gather is a single collective
    results = torch.empty(CLIP_FRAMES * (2 + 12), dtype=torch.int32, device=device)
    scores = results[: CLIP_FRAMES * 2].view(torch.float32).view(CLIP_FRAMES, 1, 2)
    counts = results[CLIP_FRAMES * 2:].view(CLIP_FRAMES, 12)
    from amatsukaze_b200 import shard
    gathered = {}
    # The score gather of a pass runs on its own stream: it waits (event) for the pass that produced `results`, copies
    # them into a snapshot, and overlaps with the next pass instead of sitting between two passes on the compute stream.
    gstream = torch.cuda.Stream(device=device) if world > 1 else None
    snap = torch.empty_like(results) if world > 1 else None
    ev_done = torch.cuda.Event() if world > 1 else None
    ev_snap = torch.cuda.Event() if world > 1 else None

    def step():
        if world > 1:
            stream.wait_event(ev_snap)                    # previous snapshot taken before results are overwritten
        ctx.scan_comb_frames(clip, [logo], prm, scores=scores, counts=counts)
        if world > 1:
            ev_done.record(stream)
            with torch.cuda.stream(gstream):
                gstream.wait_event(ev_done)
                snap.copy_(results, non_blocking=True)
                ev_snap.record(gstream)
                gathered["results"] = shard.gather_streams(snap)

    sampler = ClockSampler(local_rank)
    sampler.start()
    with torch.cuda.stream(stream):
        if world > 1:
            ev_snap.record(stream)
        for _ in range(max(args.warmup, 3)):
            step()
        stream.synchronize()
        if world > 1:
            gstream.synchronize()
            dist.barrier()
        torch.cuda.synchronize()
        l0 = ctx.launches
        ctx.kernel_timing(reset=True)
        ctx.set_kernel_timing(True)
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        sampler.active = True
        ev0.record(stream)
        for _ in range(args.steps):
            step()
        if world > 1:
            stream.wait_stream(gstream)                   # the last gather is part of the timed region
        ev1.record(stream)
        stream.synchronize()
        torch.cuda.synchronize()
        sampler.active = False
        if world > 1:
            dist.barrier()
        elapsed_ms = ev0.elapsed_time(ev1)
        comb_ms, comb_n = ctx.kernel_timing(reset=True)
        ctx.set_kernel_timing(False)
        launches = ctx.launches - l0
    if args.dump_outputs and rank == 0:
        if world > 1:                                     # every rank's results, as the last step's gather delivered them
            r = gathered["results"]
            dump_outputs(args.dump_outputs, r[:, : CLIP_FRAMES * 2].contiguous().view(torch.float32).cpu(), r[:, CLIP_FRAMES * 2:].cpu())
        else:
            dump_outputs(args.dump_outputs, scores.cpu(), counts.cpu())
    if world > 1:
        t = torch.tensor([elapsed_ms], dtype=torch.float64, device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        elapsed_ms = float(t.item())
    value = CLIP_FRAMES * world * args.steps / (elapsed_ms * 1e-3)

    # ---- end-to-end through the C ABI with HOST buffers: H2D of the clip + D2H of the results inside the timing ----
    e2e = None
    host = None
    if not args.no_e2e or (rank == 0 and not args.no_cpu):
        host = torch.empty((CLIP_FRAMES, FRAME_BYTES), dtype=torch.uint8, pin_memory=True)
        host.copy_(clip_t)
        torch.cuda.synchronize()
    if not args.no_e2e:
        hclip = ab.yv12_clip(host, W, H, CLIP_FRAMES, on_device=False)
        h_scores = np.empty((CLIP_FRAMES, 1, 2), np.float32)
        h_counts = np.empty((CLIP_FRAMES, 12), np.int32)
        with torch.cuda.stream(stream):
            ctx.scan_comb_frames(hclip, [logo], prm, scores=h_scores, counts=h_counts)     # warm-up (staging buffers)
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for _ in range(args.e2e_steps):
                ctx.scan_comb_frames(hclip, [logo], prm, scores=h_scores, counts=h_counts)   # returns after D2H + sync
            e1.record(stream)
            stream.synchronize()
            e2e_ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([e2e_ms], dtype=torch.float64, device=device)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            e2e_ms = float(t.item())
        same = bool(np.array_equal(h_scores, scores.cpu().numpy()) and np.array_equal(h_counts, counts.cpu().numpy()))
        # logo-only call on the same HOST frames: the library uploads just the logo rectangle rows (what the reference's
        # ScanFrame reads, LogoScan.hpp:1559-1566), not 3.1 MB per frame
        hs2 = np.empty((CLIP_FRAMES, 1, 2), np.float32)
        with torch.cuda.stream(stream):
            ctx.scan_frames(hclip, [logo], out=hs2)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(args.e2e_steps):
                ctx.scan_frames(hclip, [logo], out=hs2)         # blocking: returns after the D2H of the scores
            logo_e2e_s = (time.perf_counter() - t0) / args.e2e_steps
        logo_only = {"value": CLIP_FRAMES / logo_e2e_s, "unit": "frames/s", "h2d_bytes_per_step": ctx.last_h2d_bytes,
                     "full_frame_bytes_per_step": CLIP_FRAMES * FRAME_BYTES, "d2h_bytes_per_step": int(hs2.nbytes),
                     "matches_device_run": bool(np.array_equal(hs2, scores.cpu().numpy())),
                     "what": "LogoFrame::ScanFrame alone through the C ABI on host frames (ROI-only staging), wall clock per call"}
        e2e = {"value": CLIP_FRAMES * world * args.e2e_steps / (e2e_ms * 1e-3), "unit": "frames/s",
               "h2d_bytes_per_step": staged_h2d_bytes(CLIP_FRAMES, FRAME_BYTES),
               "d2h_bytes_per_step": int(h_scores.nbytes + h_counts.nbytes), "steps": args.e2e_steps,
               "host_memory": "pinned", "numa_binding": numa, "matches_device_run": same, "logo_only_host_frames": logo_only,
               "h2d_gbs_per_gpu": staged_h2d_bytes(CLIP_FRAMES, FRAME_BYTES) * args.e2e_steps / (e2e_ms * 1e-3) / 1e9,
               "note": "PCIe-bound by construction: every frame byte crosses the host link once"}

    # read-only ceiling on this GPU: a plain streaming reduction over the same 5.6 GB clip (SURVEY.md 8(d))
    with torch.cuda.stream(stream):
        read_ceiling = ctx.probe_read_gbs(clip_t, reps=3)

    sampler.stop_flag = True
    exit_code = 0
    if rank == 0:
        # roofline of the dominant kernel: algorithmic bytes = one read of every frame byte
        alg_bytes = CLIP_FRAMES * FRAME_BYTES
        avg_ms = comb_ms / max(comb_n, 1)
        achieved = alg_bytes / (avg_ms * 1e-3) / 1e9
        traffic = None
        tp = os.path.join(ROOT, "profiles", "comb_traffic.json")
        if os.path.exists(tp):
            try:
                traffic = json.load(open(tp)).get("dram_bytes_per_launch")
            except Exception:
                traffic = None
        cpu, parity = None, None
        if not args.no_cpu:
            # WHOLE-clip parity (outside every timed region) + the CPU baseline, on the host copy of the same clip
            from oracle import pyoracle as po
            threads = po.usable_cpu_threads()
            fr = host.numpy()
            cpu, sc, cn = cpu_measure(po, fr, logo_def["data"], prm.as_list(), threads)
            g_sc = scores[:, 0].cpu().numpy()
            g_cn = counts.cpu().numpy()
            s_ok = bool(np.array_equal(g_sc.view(np.uint32), sc.view(np.uint32)))
            c_ok = bool(np.array_equal(g_cn, cn))
            # the scalar (normative) form of the combing spec on a prefix, as a second witness next to the AVX2 one
            nsc = 48
            b = po.CpuBench(W, H, logo_def["data"], IMGX, IMGY, threads, MASKRATIO)
            _, _, cn_s = b.run(fr[:nsc], prm.as_list(), 2, "scalar")
            b.close()
            c_ok_scalar = bool(np.array_equal(g_cn[:nsc], cn_s))
            parity = {"frames": CLIP_FRAMES, "scores_bitexact": s_ok, "counts_equal": c_ok and c_ok_scalar,
                      "oracle": cpu["kind"], "scores_checked_against": "reference's own code (oracle/_ref), float bit patterns" if cpu["kind"] == "reference" else "C port of the reference",
                      "counts_checked_against": "combing spec: AVX2 form on all %d frames (frame 0 with prev = itself), scalar normative form on the first %d" % (CLIP_FRAMES, nsc),
                      "score_mismatches": int((g_sc.view(np.uint32) != sc.view(np.uint32)).any(axis=1).sum()),
                      "count_mismatches": int((g_cn != cn).any(axis=1).sum())}
            if not (s_ok and c_ok and c_ok_scalar):
                exit_code = 3
        secondary = None
        if not args.no_secondary and world == 1:
            del clip_t
            torch.cuda.empty_cache()
            secondary = secondary_configs(torch, ab, synth, ctx, stream, device, ["single_frame_1440", "comb_1440", "comb_p10", "logoscan_10k", "logo_analyze", "logo_scan"], peak,
                                          po=None if args.no_cpu else po)
        line = {
            "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": elapsed_ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8+f32", "data": "synthetic",
            "config": {"workload": WORKLOAD,
                       "frames_per_step_per_gpu": CLIP_FRAMES, "logo": "64x64 @(1700,60) maskratio 0.35, fades {0,1}",
                       "l2": "step input 5.6 GB per GPU is larger than the 126 MB L2 (no flush needed)",
                       "parallelism": "one independent clip per GPU" + ("; one NCCL all_gather of the results per step on a side stream" if world > 1 else "")},
            "clocks": sampler.summary(),
            "e2e": e2e,
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "kernel": "comb_ws_kernel<WsCfg<15,2>> (8-bit streaming pass)", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": alg_bytes, "avg_launch_ms": avg_ms, "launches_timed": int(comb_n),
                         "share_of_step": (comb_ms / max(elapsed_ms, 1e-9)),
                         "read_only_ceiling_gbs": read_ceiling},
            "cpu_baseline": cpu,
            "parity": parity,
            "secondary": secondary,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    ctx.close()
    if exit_code:
        sys.stderr.write("bench.py: PARITY MISMATCH against the CPU oracle (see the `parity` block)\n")
        sys.exit(exit_code)


if __name__ == "__main__":
    main()
