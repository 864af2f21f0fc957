"""The host-side C++ mirror of the reference's filter interface (amatsukaze_b200/host/filters.hpp), driven by
tests/cpp/test_filters.cpp the way CMAnalyze::logoFrame and AMTFilterSource drive the reference, checked against the
oracle and against the reference's own LogoFrame::selectLogo/writeResult (stored results; live where oracle/_ref is built)."""
import json
import os
import struct
import subprocess

import numpy as np
import pytest

import amatsukaze_b200 as ab
import ref_inputs as ri
from amatsukaze_b200 import synth, _build
from oracle import pyoracle as po

pytestmark = pytest.mark.gpu
W, H, N, IMGX, IMGY = ri.FILTERS_CLIP
REF = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "ref_cases.json")))


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


@pytest.fixture(scope="module")
def run(tmp_path_factory):
    exe = _build.build_host_test() if os.path.exists("/usr/bin/g++") else _build.HOST_TEST
    out = tmp_path_factory.mktemp("filters")
    lg, frames = ri.filters_clip()
    clip = out / "clip.amtsraw"
    with open(clip, "wb") as f:
        f.write(b"AMTSRAW1" + struct.pack("<6i", W, H, 8, N, 30000, 1001))
        f.write(frames.tobytes())
    logo_path = str(out / "logo.lgd")
    ab.Logo.create(lg["data"], 64, 64, W, H, IMGX, IMGY).save(logo_path, "No Name", 410)
    r = subprocess.run([exe, str(clip), logo_path, str(out)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    return {"out": out, "stdout": r.stdout, "lg": lg, "frames": frames}


def test_plugin_registration_and_errors(run):
    s = run["stdout"]
    assert "params: s[filter]s[outqp]b | cs[maskratio]i | ccs[logof]s[mode]i[maxfade]i" in s     # Amatsukaze.cpp:55-58
    assert "analyze vi: 64x5 8 frames" in s                                                      # LogoScan.hpp:1195-1200
    assert "expected error: Failed to read logo file (" in s                                     # LogoScan.hpp:1174
    assert "there is no function named 'NoSuchFilter'" in s
    assert s.strip().endswith("OK")


def test_logoframe_scan_select_write(run):
    out, lg, frames = run["out"], run["lg"], run["frames"]
    ev = np.fromfile(out / "eval.bin", np.float32).reshape(N, 2, 2)
    o = po.OracleLogo.create(lg["data"], 64, 64, W, H, IMGX, IMGY).deint().create_mask(0.35)
    Y, _, _ = synth.split_planes(frames, W, H)
    ref = np.stack([o.scan_frame(Y[i]) for i in range(N)])
    assert np.array_equal(_bits(ev[:, 0]), _bits(ref))
    assert np.all(ev[:, 1, 0] == 0) and np.all(ev[:, 1, 1] == -1)            # unreadable logo file -> (0,-1)
    txt = open(out / "logof.txt").read()
    assert "bestLogo=0" in run["stdout"]
    # the reference's selectLogo / writeResult on these scores (tests/golden/ref_cases.json; live where oracle/_ref is built)
    g = REF["filters_logoframe"]["fps"]["30"]
    best, ratio = g["best"], float(np.uint32(g["ratio_bits"]).view(np.float32))
    assert best == 0 and ("logoRatio=%.6f" % ratio) in run["stdout"]
    assert txt == g["text"] and len(txt.splitlines()) >= 2
    if po.ref_available():
        rp = str(out / "logof_ref.txt")
        assert po.ref_logoframe(ev, 30, rp) == (best, ratio) and open(rp).read() == txt


def test_cmanalyze_logoframe_entry(run):
    """CMAnalyze ctor -> logoFrame (CMAnalyze.hpp:25-47,273-317): picks the readable logo among the --logo list, writes
    logof0.txt for it and logof0-0.txt for the erase logo (TranscodeSetting.hpp:934-939)."""
    out = run["out"]
    assert ("cmanalyze: logopath=%s " % (out / "logo.lgd")) in run["stdout"]
    assert "cmanalyze idle: ''" in run["stdout"]
    txt = open(out / "logof.txt").read()
    assert open(out / "logof0.txt").read() == txt           # same scores, same selection as the direct LogoFrame run
    assert open(out / "logof0-0.txt").read() == txt


def test_logoframe_write_result_matches_reference_on_many_patterns(run, tmp_path):
    """selectLogo/writeResult are pure host code: the product's (tests/cpp/test_host_only.cpp driver) on the clip's scores
    under different frame rates against the reference's own implementation (LogoScan.hpp:1645-1827; results stored in
    tests/golden/ref_cases.json, and oracle/_ref live where it is built)."""
    ev = np.fromfile(run["out"] / "eval.bin", np.float32).reshape(N, 2, 2)
    exe = _build.build_host_only_test()
    for fps in ri.FILTERS_LOGOFRAME_FPS:
        g = REF["filters_logoframe"]["fps"][str(fps)]
        best, ratio = g["best"], np.uint32(g["ratio_bits"]).view(np.float32)
        assert best == 0 and 0.0 < ratio < 1.0
        if po.ref_available():
            assert po.ref_logoframe(ev, fps, str(tmp_path / ("r%d.txt" % fps))) == (best, float(ratio))
            assert open(tmp_path / ("r%d.txt" % fps)).read() == g["text"]
        sp, op = tmp_path / "s.bin", tmp_path / ("o%d.txt" % fps)
        ev.tofile(sp)
        r = subprocess.run([exe, "logoframe", str(sp), str(N), "2", str(fps), "1", str(op)], capture_output=True, text=True, timeout=120)
        assert r.returncode == 0, r.stdout + r.stderr
        assert ("bestLogo=%d " % best) in r.stdout and np.float32(float(r.stdout.split("logoRatio=")[1])) == ratio, (fps, r.stdout)
        assert open(op).read() == g["text"], fps


def test_analyze_records_and_fades(run):
    out, lg, frames = run["out"], run["lg"], run["frames"]
    rec = np.fromfile(out / "analyze.bin", np.float32).reshape(-1, 33)
    assert rec.shape[0] == 8 * ((N + 7) // 8)
    raw = po.OracleLogo.create(lg["data"], 64, 64, W, H, IMGX, IMGY)
    de, top, bot = raw.deint().create_mask(0.35), raw.field(0).create_mask(0.35), raw.field(1).create_mask(0.35)
    Y, _, _ = synth.split_planes(frames, W, H)
    ref = np.stack([po.or_analyze_frame(de, top, bot, Y[i]) for i in range(N)])
    assert np.array_equal(_bits(rec[:N]), _bits(ref))
    assert np.array_equal(_bits(rec[N:]), _bits(np.repeat(ref[-1:], rec.shape[0] - N, 0)))      # clamped tail (:1133)
    fades = np.fromfile(out / "fades.bin", np.float32).reshape(N, 2)
    exp = np.array([po.or_calc_fade2(ref, N, n) for n in range(N)], np.float32)
    assert np.array_equal(fades, exp)
    assert fades.min() == 0.0 and fades.max() == 1.0
    # with the logoframe file: uniform windows short-circuit to 0/1 (LogoScan.hpp:1326-1339)
    fl = np.fromfile(out / "fades_logof.bin", np.float32).reshape(N, 2)
    fr = np.zeros(N, int)
    el = [l.split() for l in open(out / "logof.txt").read().splitlines()]
    for i in range(0, len(el), 2):
        s0, s1, e0, e1 = int(el[i][4]), int(el[i][5]), int(el[i + 1][4]), int(el[i + 1][5])
        fr[min(N, s0):min(N, s1 + 1)] = 1
        fr[min(N, s1):min(N, e0 + 1)] = 2
        fr[min(N, e0 + 1):min(N, e1 + 1)] = 1
    for n in range(N):
        win = [fr[max(0, min(N - 1, n + i))] for i in range(-8, 9)]
        if all(v == win[0] for v in win):
            assert tuple(fl[n]) == ((1.0, 1.0) if fr[n] == 2 else (0.0, 0.0)), n
        else:
            assert tuple(fl[n]) == tuple(exp[n]), n


def test_erase_through_getframe(run):
    out, lg, frames = run["out"], run["lg"], run["frames"]
    fades = np.fromfile(out / "fades.bin", np.float32).reshape(N, 2)
    got = np.fromfile(out / "erased.bin", np.uint8).reshape(-1, W * H * 3 // 2)
    idx = list(range(0, N, 7))
    assert got.shape[0] == len(idx)
    raw = po.OracleLogo.create(lg["data"], 64, 64, W, H, IMGX, IMGY)
    changed = 0
    for k, n in enumerate(idx):
        Y, U, V = [np.ascontiguousarray(p[n]) for p in synth.split_planes(frames.copy(), W, H)]
        po.or_erase_frame(raw, Y, U, V, float(fades[n, 0]), float(fades[n, 1]))
        exp = np.concatenate([Y.ravel(), U.ravel(), V.ravel()])
        assert np.array_equal(got[k], exp), n
        changed += int(not np.array_equal(exp, frames[n]))
    assert changed > 0


def test_telecine_side_files(tmp_path_factory):
    """A 3:2 pulled-down clip through AMTCombAnalyze -> WriteTelecineFiles -> AMTDecimate / timecode reader."""
    exe = _build.HOST_TEST
    out = tmp_path_factory.mktemp("telecine")
    n = 43
    frames = synth.make_frames(0, n, W, H, mode="telecine").numpy()
    clip = out / "clip.amtsraw"
    with open(clip, "wb") as f:
        f.write(b"AMTSRAW1" + struct.pack("<6i", W, H, 8, n, 30000, 1001))
        f.write(frames.tobytes())
    lg = synth.make_logo(64, 64, seed=1)
    logo_path = str(out / "logo.lgd")
    ab.Logo.create(lg["data"], 64, 64, W, H, IMGX, IMGY).save(logo_path)
    r = subprocess.run([exe, str(clip), logo_path, str(out)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    line = [l for l in r.stdout.splitlines() if l.startswith("telecine:")][0]
    kv = dict(p.split("=") for p in line.split()[1:])
    assert int(kv["film_cycles"]) == 8                       # 43 frames = 8 full cycles + 3
    assert int(kv["decimated"]) == n - 8
    dur = [int(x) for x in open(out / "tc.duration.txt").read().split()]
    assert sum(dur) == n and dur[:5] == [1, 1, 2, 1, 1]      # synthetic pattern: frames 2,3 of every cycle are combed
    assert "decimate map: 0 1 2 4 5 6 7 9 10 11" in r.stdout
    assert int(kv["timecodes"]) == n - 8 + 1 and abs(float(kv["total_ms"]) - n * 1001 / 30) < 1e-3
    assert "[AMTDecimate] # of frames does not match. 3(" in r.stdout      # FilteredSource.hpp:653-654


def test_comb_prepass_file(run):
    out, frames = run["out"], run["frames"]
    got = np.loadtxt(out / "combstat.txt", dtype=np.int64).astype(np.int32)
    Y, U, V = synth.split_planes(frames, W, H)
    assert np.array_equal(got, po.or_comb_clip(Y, U, V, ab.default_comb_params().as_list()))
