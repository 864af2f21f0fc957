"""Seeded inputs of the tests that compare with the reference's stored results (tests/golden/ref_cases.json and
ref_sizes.json).  tests/golden/gen_golden.py builds those files from these same functions, so the tests and the golden
data cannot drift apart: a changed input changes the digests and the tests fail until the golden data is regenerated."""
import numpy as np
import torch

from amatsukaze_b200 import synth

# ---- tests/test_oracle.py ----
LOGO_FRAME = (320, 200, 100, 60)                    # frame width, height and the logo position of logo_cases()


def logo_cases():
    """Random logos / planes beyond logo_golden.json: (case, w, h, data, ratio, maxv, planes) for 8- and 16-bit samples, odd
    sizes and a logo whose mask spills into zero-variance pixels."""
    rng = np.random.default_rng(7)
    fw, fh, _, _ = LOGO_FRAME
    for case, (w, h, ratio, bitsps) in enumerate(((64, 64, 0.35, 8), (48, 40, 0.9, 8), (64, 32, 0.35, 10), (32, 64, 0.1, 8))):
        data = synth.make_logo(w, h, seed=case)["data"].copy()
        if case == 1:
            data[: w * h][(rng.random(w * h) < 0.3)] *= 1.0      # keep flat areas: high maskratio forces border picks
        maxv = float((1 << bitsps) - 1)
        planes = [rng.integers(16, 236, (fh, fw), dtype=np.uint8) if bitsps == 8 else rng.integers(64, 940, (fh, fw)).astype(np.uint16)
                  for _ in range(4)]
        yield case, w, h, data, ratio, maxv, planes


def logoscan_frames():
    """60 (y, u, v) 24x16 ROIs for a LogoScan with thy 10: a brighter logo block on a noisy base, every 7th frame with a
    pixel that breaks the flat-border test."""
    rng = np.random.default_rng(11)
    for i in range(60):
        base = int(rng.integers(30, 200))
        y = (base + rng.integers(-3, 4, (16, 24))).astype(np.uint8)
        if i % 7 == 0:
            y[0, 3] = 255
        u = (128 + rng.integers(-2, 3, (8, 12))).astype(np.uint8)
        v = (128 + rng.integers(-2, 3, (8, 12))).astype(np.uint8)
        y[4:12, 6:18] = np.clip(y[4:12, 6:18].astype(int) + 40, 0, 255).astype(np.uint8)
        yield y, u, v


DELOGO_FADES = (0.0, 0.1, 0.3, 0.5, 0.9, 1.0)


def delogo_and_calc_fade2_cases():
    """([(dtype, maxv, w, h, logopitch, imgpitch, img, A, B)], [(N, records)]): Delogo rectangles incl. the per-field pitches
    (logopitch 2w, imgpitch 2*pitch), and analyze records with sudden appear / disappear patterns so that both branches of
    CalcFade2 (LogoScan.hpp:1295-1314) are taken."""
    rng = np.random.default_rng(11)
    delogo = []
    for dtype, maxv in ((np.uint8, 255.0), (np.uint16, 1023.0)):
        for (w, h, lp, ip) in ((64, 64, 64, 96), (32, 16, 64, 200), (7, 5, 7, 7)):
            img = rng.integers(0, int(maxv) + 1, size=(h, ip)).astype(dtype)
            A = rng.uniform(0.8, 1.6, size=h * lp).astype(np.float32)
            B = rng.uniform(-0.6, 0.1, size=h * lp).astype(np.float32)
            delogo.append((dtype, maxv, w, h, lp, ip, img, A, B))
    fade2 = []
    for N in (1, 5, 8, 9, 23, 64, 101):
        rec = rng.uniform(0.0, 1.0, size=(N, 33)).astype(np.float32)
        for k in range(N):
            rec[k, : 11] += np.abs(np.arange(11) - (0 if (k // 7) % 2 == 0 else 10)) * np.float32(0.5)
        fade2.append((N, rec))
    return delogo, fade2


def mergefield_cases():
    """(w, h, top, bottom): two packed planar 4:2:0 frames per size; heights are multiples of 4 because Copy1 writes row
    pairs of the chroma planes too."""
    rng = np.random.default_rng(5)
    for (w, h) in ((16, 8), (208, 72), (64, 36)):
        n = w * h + 2 * (w // 2) * (h // 2)
        yield w, h, rng.integers(0, 256, n).astype(np.uint8), rng.integers(0, 256, n).astype(np.uint8)


def to_nv12(a, w, h):
    """A packed planar 4:2:0 frame with its chroma interleaved (NV12)."""
    ysz, csz = w * h, (w // 2) * (h // 2)
    return np.concatenate([a[:ysz], np.stack([a[ysz:ysz + csz], a[ysz + csz:]], axis=1).reshape(-1)])


def drivers_clip():
    """(w, h, imgx, imgy, logo, frames): the clip of the GetFrameT / ScanFrame driver test (13 frames: two analyze frames,
    the second clamped at the clip end)."""
    w, h, imgx, imgy, n = 256, 128, 160, 32, 13
    lg = synth.make_logo(64, 64)
    return w, h, imgx, imgy, lg, synth.make_frames(40, n, w, h, device="cpu", logo=lg, imgx=imgx, imgy=imgy, logo_period=12).numpy()


DRIVER_SCAN_FRAMES = (0, 5, 12)


# ---- tests/test_host_only.py ----
LOGOFRAME_FPS = ((24000, 1001), (30000, 1001), (60000, 1001), (25, 1))
LOGOFRAME_CASES = [
    [[(100, 400)], [(0, 0)]],                                   # one section, second logo never present
    [[(0, 250), (400, 700)], [(50, 120)]],                      # starts and ends inside a section
    [[(60, 90), (130, 170), (300, 650)], [(0, 700)]],           # short sections, always-on competitor
    [[(0, 0)], [(0, 0)]],                                       # nothing anywhere
    [[(0, 700)], [(200, 500)]],                                 # everything
    [[(200, 210), (215, 500)], [(10, 20)]],                     # a gap shorter than the filters
]


def score_track(rng, n, on_ranges, noise=0.08, flicker=0.0):
    """(n, 2) corr0/corr1 as ScanFrame produces them: logo present -> corr0 high, corr1 ~ 0; absent -> corr0 ~ 0, corr1 < 0."""
    on = np.zeros(n, bool)
    for a, b in on_ranges:
        on[a:b] = True
    if flicker:
        on ^= rng.random(n) < flicker
    c0 = np.where(on, 0.8, 0.0) + rng.normal(0, noise, n)
    c1 = np.where(on, 0.0, -0.8) + rng.normal(0, noise, n)
    return np.stack([c0, c1], 1).astype(np.float32)


def logoframe_tracks(fps):
    """(case, flicker, scores (700, 2 logos, 2)) for every LOGOFRAME_CASES entry, with and without flicker."""
    rng = np.random.default_rng(fps[0])
    for ci, (a, b) in enumerate(LOGOFRAME_CASES):
        for flicker in (0.0, 0.03):
            yield ci, flicker, np.stack([score_track(rng, 700, a, flicker=flicker), score_track(rng, 700, b, flicker=flicker)], 1)


def sidefile_inputs():
    """(timecode file texts, duration lists): v2 timecodes on 60/120/240 fps grids and irregular, with and without the total
    line, CRLF and comments, plus edge cases (empty file, one stamp, total line only, total line with trailing text)."""
    rng = np.random.default_rng(3)
    texts = []
    for grid in (60, 120, 240, 0):
        t, stamps = 0.0, []
        for _ in range(int(rng.integers(2, 90))):
            stamps.append(int(round(t)))
            t += (1001.0 / grid * 1000.0 / 1000.0 * int(rng.integers(1, 4)) * (1000.0 / 1000.0)) if grid else float(rng.integers(5, 80))
        body = "# timecode format v2\n" + "".join("%d\n" % v for v in stamps)
        texts += [body + "# total: %.3f\n" % (t / 1000.0), body, body + "\r\n#comment\n\n"]
    texts += ["", "17\n", "# total: 12.5\n", "5\n9\n# total: 1.0 trailing\n33\n"]
    durations = [[int(v) for v in rng.integers(1, 4, size=int(rng.integers(1, 60)))] for _ in range(8)]
    return texts, durations


def erase_fades_inputs():
    """(n, maxfade, analyze records (n, 33), logoframe elements ((start, fadein0, fadein1), (end, fadeout0, fadeout1)))."""
    rng = np.random.default_rng(11)
    return 120, 16, rng.normal(0.0, 0.5, (120, 33)).astype(np.float32), [((22, 20, 26), (58, 55, 61)), ((90, 88, 93), (118, 115, 119))]


def logoframe_file(elems):
    """A logoframe file (LogoScan.hpp:1818-1819 format)."""
    return "".join("%6d S 0 ALL %6d %6d\n%6d E 0 ALL %6d %6d\n" % (*s, *e) for s, e in elems)


# ---- tests/test_host_filters.py, tests/test_gpu_parity.py ----
FILTERS_CLIP = (256, 128, 61, 160, 32)               # W, H, frames, logo position of filters_clip()


def filters_clip():
    """(logo, frames) of the host filter test's 61-frame clip."""
    W, H, N, IMGX, IMGY = FILTERS_CLIP
    lg = synth.make_logo(64, 64, seed=1)
    return lg, synth.make_frames(35, N, W, H, logo=lg, imgx=IMGX, imgy=IMGY, logo_period=40).numpy()


FILTERS_LOGOFRAME_FPS = (24, 30, 60)
WEAVE = (208, 72, 6, [0, 1, 2, 3, 4, 5], [1, 2, 3, 4, 5, 5])        # w, h, frames, top and bottom source of each output frame


def weave_frames(device="cpu"):
    w, h, n, _, _ = WEAVE
    return synth.make_frames(0, n, w, h, device=device, mode="interlaced")


# ---- tests/test_gpu_parity_sizes.py ----
def gen_frames(n0, n, w, h, device="cpu", chunk=10, **kw):
    """Frames n0..n0+n-1 generated in chunks (the generator is integer-only: CPU and CUDA frames are identical)."""
    out = torch.empty((n, w * h * 3 // 2), dtype=torch.uint8, device=device)
    for k in range(0, n, chunk):
        m = min(chunk, n - k)
        synth.make_frames(n0 + k, m, w, h, device=device, out=out[k:k + m], **kw)
    return out


SCAN_1440 = (1440, 1080, 16, 1280, 64)              # configs[0] geometry: w, h, frames, logo position


def scan_1440_frames(logo, device="cpu"):
    w, h, n, imgx, imgy = SCAN_1440
    return gen_frames(35, n, w, h, device, logo=logo, imgx=imgx, imgy=imgy, logo_period=16)


WHOLE_CLIP = (1920, 1080, 1000, 1700, 60)           # 1000 frames of the bench clip: w, h, frames, logo position


def whole_clip_frames(logo, device="cpu"):
    w, h, n, imgx, imgy = WHOLE_CLIP
    return gen_frames(0, n, w, h, device, logo=logo, imgx=imgx, imgy=imgy)


LOGOSCAN_10K = (1920, 1080, 10000)                  # configs[3]: w, h, frames
LOGOSCAN_10K_ROIS = ((1700, 60, 64, 64), (1600, 60, 256, 128))


def logoscan_10k_frames(k, count, logo, device="cpu", out=None):
    """Frames k..k+count-1 of the flat 10000-frame LogoScan clip."""
    w, h, _ = LOGOSCAN_10K
    return synth.make_frames(k, count, w, h, seed=0x5EED0007, device=device, mode="flat", logo=logo, imgx=1700, imgy=60, out=out)
