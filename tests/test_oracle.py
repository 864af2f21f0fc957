"""CPU tests of the checker itself: the plain-C oracle (oracle/amtk_oracle.c) must reproduce
  (1) the committed golden vectors the REFERENCE'S OWN code produced (tests/golden/logo_golden.json), always;
  (2) the reference's results on further cases, stored in tests/golden/ref_cases.json, and the reference's own compiled
      code (oracle/_ref) live, when that library is present.
All float comparisons are on bit patterns."""
import ctypes as C
import hashlib
import json
import os

import numpy as np
import pytest

import ref_inputs as ri
from amatsukaze_b200 import synth
from oracle import pyoracle as po

GOLD = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "logo_golden.json")))
REF = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "ref_cases.json")))
W, H, IMGX, IMGY = 256, 128, 160, 32


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32).ravel().tolist()


def digest(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


@pytest.fixture(scope="module")
def data():
    lg = synth.make_logo(64, 64, seed=1)
    frames = synth.make_frames(40, 24, W, H, seed=0x5EED0001, logo=lg, imgx=IMGX, imgy=IMGY, logo_period=20).numpy()
    raw = po.OracleLogo.create(lg["data"], 64, 64, W, H, IMGX, IMGY)
    logos = {"raw": raw, "deint": raw.deint().create_mask(0.35), "top": raw.field(0).create_mask(0.35),
             "bot": raw.field(1).create_mask(0.35), "deint10": raw.deint().create_mask(0.1)}
    return lg, frames, logos


def test_corr5x5_avx_tree_matches_golden():
    g = GOLD["corr5x5"]
    rng = np.random.default_rng(g["seed"])
    Y = np.concatenate([(rng.random(20 * 20) * 255).astype(np.float32), np.zeros(8, np.float32)])
    K = np.concatenate([rng.standard_normal(25).astype(np.float32), np.zeros(8, np.float32)])
    L = po.oracle_lib()
    sums, avgs, scalar = [], [], []
    for y in range(2, 18):
        for x in range(2, 18):
            a = C.c_float()
            sums.append(L.amtk_or_corr5x5(K.ctypes.data_as(po.c_float_p), Y.ctypes.data_as(po.c_float_p), x, y, 20, C.byref(a)))
            avgs.append(a.value)
            scalar.append(L.amtk_or_corr5x5_scalar_order(K.ctypes.data_as(po.c_float_p), Y.ctypes.data_as(po.c_float_p), x, y, 20, None))
    assert bits(sums) == g["sum_bits"] and bits(avgs) == g["avg_bits"]
    # the scalar summation order is NOT what the reference runs on AVX hosts and differs in the last bits (SURVEY 0.6)
    assert bits(scalar) != g["sum_bits"]
    assert np.allclose(scalar, sums, rtol=2e-3, atol=1e-2)


def test_tables_match_golden(data):
    _, _, logos = data
    for name, t in GOLD["tables"].items():
        l = logos[name]
        ny = l.s.w * l.s.h
        assert l.s.maskpixels == t["maskpixels"] and l.s.count == t["count"]
        assert bits([l.s.blackScore])[0] == t["black_bits"]
        assert digest(l.data()[:2 * ny]) == t["ab_sha"]
        assert digest(l.mask()) == t["mask_sha"]
        assert digest(l.kernels()) == t["kernels_sha"]
        assert digest(l.scales()) == t["scales_sha"]


def test_scan_and_analyze_match_golden(data):
    _, frames, logos = data
    Y, _, _ = synth.split_planes(frames, W, H)
    for i in range(frames.shape[0]):
        assert bits(logos["deint"].scan_frame(Y[i])) == GOLD["scan_frame_bits"][i]
    for k, i in enumerate(GOLD["analyze_frames"]):
        assert bits(po.or_analyze_frame(logos["deint"], logos["top"], logos["bot"], Y[i])) == GOLD["analyze_bits"][k]
    on = np.array([np.array(b, np.uint32).view(np.float32)[0] for b in GOLD["scan_frame_bits"]])
    assert on.max() > 0.8 and on.min() < 0.2          # the fixture covers logo present AND absent


def test_fade_sweep_matches_golden(data):
    _, frames, logos = data
    Y, _, _ = synth.split_planes(frames, W, H)
    de = np.zeros(64 * 64 + 8, np.float32)
    roi = np.ascontiguousarray(Y[12])
    po.oracle_lib().amtk_or_deint_y_u8(de.ctypes.data_as(po.c_float_p), roi.reshape(-1)[IMGX + IMGY * W:].ctypes.data_as(po.c_u8_p), W, 64, 64)
    got = [logos["deint10"].evaluate(de, 255.0, np.float32(0.1) * np.float32(fi)) for fi in range(20)]
    assert bits(got) == GOLD["fade_sweep_bits"]


def test_logoscan_matches_golden():
    flat = synth.make_frames(0, 40, 128, 96, seed=0x5EED0004, mode="flat", logo=synth.make_logo(32, 32, seed=3), imgx=64, imgy=32).numpy()
    fy, fu, fv = synth.split_planes(flat, 128, 96)
    sc = po.OracleScan(32, 32, 12)
    valid = [sc.add_frame(fy[i][32:64, 64:96], fu[i][16:32, 32:48], fv[i][16:32, 32:48]) for i in range(flat.shape[0])]
    g = GOLD["scan"]
    assert valid == g["valid"] and sc.nframes == g["nframes"] and 0 < sc.nframes < len(valid)
    assert digest(sc.sums()) == g["sums_sha"]
    lg = sc.get_logo(255, clean=False)
    assert digest(lg) == g["logo_sha"] and bits(lg[:16]) == g["logo_head_bits"]
    assert digest(sc.get_logo(255, clean=True)) == g["logo_clean_sha"]


def test_logoscan_insufficient_frames_returns_none():
    sc = po.OracleScan(16, 16, 12)
    assert sc.get_logo(255) is None      # 0 frames -> NaN slopes -> the reference returns nullptr (LogoScan.hpp:391,503)


def _port_logo_tables(o, planes, maxv):
    return {"count": o.s.count, "maskpixels": o.s.maskpixels, "mask_sha": digest(o.mask()), "kernels_sha": digest(o.kernels()),
            "scales_sha": digest(o.scales()), "black_bits": bits([o.s.blackScore])[0],
            "scan_bits": [bits(o.scan_frame(p, maxv=maxv)) for p in planes]}


def test_oracle_equals_reference_live():
    """Random logos / frames beyond the golden set, incl. 16-bit samples, odd sizes and a logo whose mask
    spills into zero-variance pixels (count < maskpixels, SURVEY 8 quirks).  The reference's results are stored in
    tests/golden/ref_cases.json; where oracle/_ref is built, the reference is also run live."""
    fw, fh, ix, iy = ri.LOGO_FRAME
    for case, w, h, data, ratio, maxv, planes in ri.logo_cases():
        o = po.OracleLogo.create(data, w, h, fw, fh, ix, iy).deint().create_mask(ratio)
        got = _port_logo_tables(o, planes, maxv)
        assert got == REF["logos"][case], case
        if po.ref_available():
            r = po.RefLogo.create(data, w, h, fw, fh, ix, iy).deint().create_mask(ratio)
            assert np.array_equal(r.mask(), o.mask()) and r.visited_count() == o.s.count
            assert np.array_equal(r.kernels().view(np.uint32), o.kernels().view(np.uint32))
            assert np.array_equal(r.scales().view(np.uint32), o.scales().view(np.uint32))
            assert [bits(po.ref_scan_frame(r, p, maxv)) for p in planes] == got["scan_bits"]
        if case == 1:
            assert o.s.count < o.s.maskpixels          # the quirk case really happened


def test_oracle_logoscan_equals_reference_live():
    ro = po.RefScan(24, 16, 10) if po.ref_available() else None
    oo = po.OracleScan(24, 16, 10)
    g = REF["logoscan"]
    for i, (y, u, v) in enumerate(ri.logoscan_frames()):
        assert oo.add_frame(y, u, v) == g["valid"][i]
        if ro is not None:
            assert ro.add_frame(y, u, v) == g["valid"][i]
    assert oo.nframes == g["nframes"]
    assert digest(oo.sums()) == g["sums_sha"]
    for k, clean in enumerate((False, True)):
        b = oo.get_logo(255, clean)
        assert (None if b is None else digest(b)) == g["logo_sha"][k]
    if ro is not None:
        assert ro.nframes == oo.nframes and np.array_equal(ro.sums(), oo.sums())
        for clean in (False, True):
            a, b = ro.get_logo(255, clean), oo.get_logo(255, clean)
            assert (a is None) == (b is None)
            if a is not None:
                assert np.array_equal(a.view(np.uint32), b.view(np.uint32))


def test_port_delogo_and_calcfade2_equal_the_reference_code_live():
    """Round 2: AMTEraseLogo::Delogo and CalcFade2 (LogoScan.hpp:1248-1315) are compiled from the reference's own lines into
    oracle/_ref; the plain-C port (which the GPU erase kernel and the product's amtk_calc_fade2 are tested against) must
    reproduce them exactly: pixel bytes for Delogo (rounding, clamping, per-field pitches), the selected fades for
    CalcFade2 incl. the double-offset quirk (:1273-1275) and the clip-end clamps.  The reference's results are stored in
    tests/golden/ref_cases.json and also computed live where oracle/_ref is built."""
    live = po.ref_has_erase()
    delogo, fade2 = ri.delogo_and_calc_fade2_cases()
    want = iter(REF["delogo_sha"])
    for dtype, maxv, w, h, lp, ip, img, A, B in delogo:
        for fade in ri.DELOGO_FADES:
            a = img.copy()
            po.or_delogo(a, A, B, fade, maxv, logopitch=lp, imgpitch=ip, w=w, h=h)
            assert digest(a) == next(want), (dtype, w, h, fade)
            if live:
                b = img.copy()
                po.ref_delogo(b, A, B, fade, maxv, logopitch=lp, imgpitch=ip, w=w, h=h)
                assert np.array_equal(a, b), (dtype, w, h, fade)
            assert fade == 0.0 or not np.array_equal(a, img)
    for N, rec in fade2:
        want_n = np.array(REF["calc_fade2_bits"][str(N)], np.uint32).view(np.float32).reshape(N, 2)
        took = set()
        for n in range(N):
            got = po.or_calc_fade2(rec, N, n)
            assert bits(got) == bits(want_n[n]), (N, n, got, want_n[n])
            if live:
                assert po.ref_calc_fade2(rec, N, n) == got, (N, n)
            took.add(bool(want_n[n, 0] == want_n[n, 1]))
        if N >= 23:
            assert took == {True, False}


def test_reference_mergefield_is_the_even_odd_row_weave_live():
    """AMTSource::MergeField / Copy1 / Copy2 compiled from the reference's own lines (AMTSource.hpp:291-355): even rows of
    every plane from `top`, odd rows from `bottom`, NV12 chroma de-interleaved -- the statement the GPU weave kernel
    (amtk_weave_frames) is tested against on the device.  The reference's outputs are stored as digests in
    tests/golden/ref_cases.json and also computed live where oracle/_ref is built."""
    live = po.ref_has_mergefield()
    for k, (w, h, t, b) in enumerate(ri.mergefield_cases()):
        ysz, cw, ch = w * h, w // 2, h // 2
        exp = t.copy()
        for (o, rows, cols) in ((0, h, w), (ysz, ch, cw), (ysz + cw * ch, ch, cw)):
            exp[o:o + rows * cols].reshape(rows, cols)[1::2] = b[o:o + rows * cols].reshape(rows, cols)[1::2]
        g = REF["mergefield"][k]
        assert (g["w"], g["h"]) == (w, h)
        assert digest(exp) == g["planar_sha"] and digest(exp) == g["nv12_sha"], (w, h)
        if live:
            assert np.array_equal(po.ref_merge_field(t, b, w, h), exp)
            assert np.array_equal(po.ref_merge_field(ri.to_nv12(t, w, h), ri.to_nv12(b, w, h), w, h, nv12=True), exp)


def test_reference_frame_drivers_equal_their_restated_compositions_live():
    """AMTAnalyzeLogo::GetFrameT (LogoScan.hpp:1119-1161) and LogoFrame::ScanFrame (:1543-1568) compiled from the reference's
    own lines (results stored in tests/golden/ref_cases.json): the compositions the parity tests use (DeintY, CopyY and
    EvaluateLogo called in the order those functions call them) give the same bits, including the source-frame clamp at the
    clip end (:1133), the |.| of every evaluation, and the (0, -1) result for invalid or wrong-sized logos (:1551-1558).
    Checked for the port's compositions (or_analyze_frame / scan_frame) always, and where oracle/_ref is built for the
    reference's (ref_analyze_frame / ref_scan_frame, the oracle of tests/test_gpu_parity_sizes.py there) against the live
    drivers."""
    w, h, imgx, imgy, lg, fr = ri.drivers_clip()
    N = fr.shape[0]
    raw = po.OracleLogo.create(lg["data"], 64, 64, w, h, imgx, imgy)
    de, top, bot = raw.deint().create_mask(0.35), raw.field(0).create_mask(0.35), raw.field(1).create_mask(0.35)
    Y = fr[:, : w * h].reshape(N, h, w)
    g = REF["drivers"]
    for n in range((N + 7) // 8):
        want = np.stack([po.or_analyze_frame(de, top, bot, Y[min(N - 1, 8 * n + i)]) for i in range(8)])
        assert bits(want) == g["getframe_bits"][n], n
    assert g["scanframe_frames"] == list(ri.DRIVER_SCAN_FRAMES)
    for k, i in enumerate(ri.DRIVER_SCAN_FRAMES):
        got = np.array(g["scanframe_bits"][k], np.uint32).view(np.float32).reshape(3, 2)
        assert bits(got[0]) == bits(de.scan_frame(Y[i]))
        assert tuple(got[1]) == (0.0, -1.0) and tuple(got[2]) == (0.0, -1.0)
    if po.ref_has_drivers():
        rraw = po.RefLogo.create(lg["data"], 64, 64, w, h, imgx, imgy)
        rde, rtop, rbot = rraw.deint().create_mask(0.35), rraw.field(0).create_mask(0.35), rraw.field(1).create_mask(0.35)
        for n in range((N + 7) // 8):
            got = po.ref_analyze_getframe(rde, rtop, rbot, fr, w, h, n)
            want = np.stack([po.ref_analyze_frame(rde, rtop, rbot, Y[min(N - 1, 8 * n + i)]) for i in range(8)])
            assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), n
            assert bits(got) == g["getframe_bits"][n], n
        other = po.RefLogo.create(lg["data"], 64, 64, w + 16, h, imgx, imgy).deint().create_mask(0.35)      # made for another frame size
        for k, i in enumerate(ri.DRIVER_SCAN_FRAMES):
            got = po.ref_scan_frame_code([rde, None, other], fr[i], w, h)
            assert np.array_equal(got[0].view(np.uint32), po.ref_scan_frame(rde, Y[i]).view(np.uint32))
            assert tuple(got[1]) == (0.0, -1.0) and tuple(got[2]) == (0.0, -1.0)
            assert bits(got) == g["scanframe_bits"][k]


def test_erase_and_weave_golden_from_the_reference_code(tmp_path):
    """Committed golden vectors produced by the reference's own Delogo / CalcFade2 / CalcFade + ReadLogoFrameFile / MergeField
    (tests/golden/gen_golden.py, round 2): the C port, the product's host-side amtk_calc_fade2 and the even/odd-row weave
    statement reproduce them -- also where /root/reference is absent."""
    import amatsukaze_b200 as ab
    g = GOLD["erase"]
    rng = np.random.default_rng(g["seed"])
    it = iter(g["delogo"])
    for dtype, maxv in (("uint8", 255.0), ("uint16", 1023.0)):
        for (w, h, lp, ip) in ((64, 64, 64, 96), (32, 16, 64, 200)):
            img = rng.integers(0, int(maxv) + 1, size=(h, ip)).astype(dtype)
            A = rng.uniform(0.8, 1.6, size=h * lp).astype(np.float32)
            B = rng.uniform(-0.6, 0.1, size=h * lp).astype(np.float32)
            for fade in (0.1, 0.5, 1.0):
                e = next(it)
                assert (e["dtype"], e["w"], e["h"], e["fade"]) == (dtype, w, h, fade)
                a = img.copy()
                po.or_delogo(a, A, B, fade, maxv, logopitch=lp, imgpitch=ip, w=w, h=h)
                assert digest(a) == e["sha"], e
    c2 = g["calc_fade2"]
    N = c2["n"]
    rng = np.random.default_rng(c2["seed"])
    rec = rng.uniform(0.0, 1.0, size=(N, 33)).astype(np.float32)
    for k in range(N):
        rec[k, :11] += np.abs(np.arange(11) - (0 if (k // 7) % 2 == 0 else 10)) * np.float32(0.5)
    want = np.array(c2["fades_bits"], np.uint32).view(np.float32).reshape(N, 2)
    assert bits(np.array([po.or_calc_fade2(rec, N, n) for n in range(N)], np.float32)) == c2["fades_bits"]
    assert bits(np.array([ab.calc_fade2(rec, N, n) for n in range(N)], np.float32)) == c2["fades_bits"]        # product (host code, no GPU)
    # CalcFade with a logoframe file: uniform +-maxfade/2 neighbourhoods take 0 / 1, the rest CalcFade2 (LogoScan.hpp:1317-1341)
    cf = g["calc_fade"]
    state = np.array(cf["state"], np.int32)
    half = cf["maxfade"] >> 1
    exp = np.zeros((N, 2), np.float32)
    for i in range(N):
        win = state[np.clip(np.arange(i - half, i + half + 1), 0, N - 1)]
        exp[i] = ((1.0, 1.0) if state[i] == 2 else (0.0, 0.0)) if np.all(win == win[0]) else want[i]
    assert bits(exp) == cf["fades_bits"]
    assert set(state.tolist()) == {0, 1, 2}
    # MergeField: even rows from top, odd rows from bottom, every plane
    m = GOLD["mergefield"]
    w, h = m["w"], m["h"]
    rng = np.random.default_rng(m["seed"])
    msz = w * h * 3 // 2
    t = rng.integers(0, 256, msz).astype(np.uint8)
    b = rng.integers(0, 256, msz).astype(np.uint8)
    out = t.copy()
    for (o, rows, cols) in ((0, h, w), (w * h, h // 2, w // 2), (w * h + (w // 2) * (h // 2), h // 2, w // 2)):
        out[o:o + rows * cols].reshape(rows, cols)[1::2] = b[o:o + rows * cols].reshape(rows, cols)[1::2]
    assert digest(out) == m["sha"]
