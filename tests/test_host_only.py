"""Host-side logic of the filter mirror that needs no device (tests/cpp/test_host_only.cpp): LogoFrame::selectLogo /
writeResult against the reference's own code (LogoScan.hpp:1645-1827; results stored in tests/golden/ref_cases.json, and
oracle/_ref live where it is built), AMTEraseLogo's
logoframe state machine + fade selection against the oracle's CalcFade2, AMTDecimate, the timecode reader and the
telecine side files.  CPU suite."""
import json
import os
import subprocess

import numpy as np
import pytest

import amatsukaze_b200 as ab
import ref_inputs as ri
from amatsukaze_b200 import _build, synth
from oracle import pyoracle as po

REF = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "ref_cases.json")))


@pytest.fixture(scope="module")
def exe():
    return _build.build_host_only_test()


def run(exe, *args, ok=(0,)):
    r = subprocess.run([exe, *[str(a) for a in args]], capture_output=True, text=True, timeout=120)
    assert r.returncode in ok, (r.returncode, r.stdout, r.stderr)
    return r


@pytest.mark.parametrize("fps", ri.LOGOFRAME_FPS)
def test_logoframe_select_and_write_match_reference(exe, tmp_path, fps):
    """The product's LogoFrame::selectLogo / writeResult against the reference's results on the same score tracks (stored in
    tests/golden/ref_cases.json; also computed live where oracle/_ref is built)."""
    n = 700
    want = iter(REF["logoframe"]["%d/%d" % fps])
    for ci, flicker, ev in ri.logoframe_tracks(fps):              # ev: (n, 2 logos, 2)
            sp, op, rp = tmp_path / "s.bin", tmp_path / "o.txt", tmp_path / "r.txt"
            ev.tofile(sp)
            r = run(exe, "logoframe", sp, n, 2, fps[0], fps[1], op)
            g = next(want)
            best, ratio, text = g["best"], np.uint32(g["ratio_bits"]).view(np.float32), g["text"]
            if po.ref_available():
                live = po.ref_logoframe(ev, int(round(fps[0] / fps[1])), str(rp))
                assert live == (best, float(ratio)) and open(rp).read() == text, (ci, flicker)
            assert ("bestLogo=%d " % best) in r.stdout, (ci, flicker, r.stdout, best)
            got_ratio = float(r.stdout.split("logoRatio=")[1])
            assert np.float32(got_ratio) == ratio
            assert open(op).read() == text, (ci, flicker)


def test_timecode_reader(exe, tmp_path):
    # explicit total, comments, CRLF
    p = tmp_path / "a.txt"
    p.write_bytes(b"# timecode format v2\r\n0\r\n33\r\n67\r\n\r\n# total: 0.1001\r\n999\r\n")
    out = run(exe, "timecode", p).stdout.split()
    assert out[:3] == ["ok=1", "n=4", "fps=0"] or out[:2] == ["ok=1", "n=4"]
    assert [float(x) for x in out[3:]] == [0.0, 33.0, 67.0, pytest.approx(100.1)]
    # no total: the end time is extrapolated from the last two stamps
    p.write_text("0\n42\n83\n")
    out = run(exe, "timecode", p).stdout.split()
    assert [float(x) for x in out[3:]] == [0.0, 42.0, 83.0, 124.0]
    # a single stamp: one 60 fps frame is appended
    p.write_text("500\n")
    out = run(exe, "timecode", p).stdout.split()
    assert [float(x) for x in out[3:]] == [500.0, pytest.approx(500 + 1000 / 60, abs=1e-5)]
    # stamps on the 120000/1001 grid are recognised as 120 fps VFR timing (FilteredSource.hpp:190-211)
    grid = [int(round(k * 1001 / 120.0)) for k in (0, 5, 9, 14, 18, 23, 27, 32, 36)]
    p.write_text("".join("%d\n" % t for t in grid))
    assert "fps=120" in run(exe, "timecode", p).stdout or "fps=240" in run(exe, "timecode", p).stdout
    # missing file / empty file
    assert "ok=0" in run(exe, "timecode", tmp_path / "nope.txt").stdout
    p.write_text("")
    assert "ok=1 n=0" in run(exe, "timecode", p).stdout


def test_decimate_map_and_mismatch(exe, tmp_path):
    d = tmp_path / "d.txt"
    d.write_text("".join("%d\n" % v for v in [1, 1, 2, 1] * 3 + [1, 1]))
    out = run(exe, "decimate", d, 17).stdout
    assert out.startswith("frames=14 map: 0 1 2 4 5 6 7 9 10 11 12 14 15 16")
    r = run(exe, "decimate", d, 18, ok=(4,))                       # AMTSource.hpp-style error text
    assert "# of frames does not match. 17(" in r.stdout and "vs 18(source clip)" in r.stdout
    r = run(exe, "decimate", tmp_path / "missing.txt", 5, ok=(4,))
    assert "failed to open" in r.stdout


def test_sidefile_readers_equal_the_reference_code(exe, tmp_path):
    """The product's TimecodeFile and AMTDecimate (host/filters.hpp) against the reference's OWN readTimecodeFile + base-fps
    estimate and AMTDecimate constructor/GetFrame (FilteredSource.hpp:163-188,197-210,645-660,663-666; their results on these
    files are stored in tests/golden/ref_cases.json and also computed live where oracle/_ref is built): same time codes
    (compared at the driver's printed 1e-6 ms resolution), same vfrTimingFps, same frame map, same mismatch message; edge
    cases: empty file, one stamp, total line with trailing text, CRLF, comments, no total line."""
    live = po.ref_has_sidefiles()
    g = REF["sidefiles"]
    cases, durations = ri.sidefile_inputs()
    assert len(cases) == len(g["timecode"])
    for k, text in enumerate(cases):
        p = tmp_path / ("tc%d.txt" % k)
        p.write_bytes(text.encode())
        out = run(exe, "timecode", p).stdout.split()
        codes, fps = g["timecode"][k]["codes"], g["timecode"][k]["fps"]
        if live:
            assert po.ref_read_timecode(p) == (codes, fps), k
        assert out[0] == "ok=1" and out[1] == "n=%d" % len(codes) and out[2] == "fps=%d" % fps, (k, out[:3], len(codes), fps)
        assert [float(x) for x in out[3:]] == [float("%.6f" % c) for c in codes], k
    assert "ok=0" in run(exe, "timecode", tmp_path / "missing.txt").stdout
    if live:
        assert po.ref_read_timecode(tmp_path / "missing.txt") is None
    for k, dur in enumerate(durations):
        d = tmp_path / ("dur%d.txt" % k)
        d.write_text("".join("%d\n" % v for v in dur))
        want, err = g["decimate"][k]["map"], g["decimate"][k]["mismatch_error"]
        if live:
            assert po.ref_decimate_map(d, sum(dur)) == want
            with pytest.raises(RuntimeError) as ei:
                po.ref_decimate_map(d, sum(dur) + 1)
            assert str(ei.value).replace(str(d), "<path>") == err
        out = run(exe, "decimate", d, sum(dur)).stdout
        assert out.split("map:")[0].strip() == "frames=%d" % len(want) and [int(x) for x in out.split("map:")[1].split()] == want
        r = run(exe, "decimate", d, sum(dur) + 1, ok=(4,))
        assert "[AMTDecimate] # of frames does not match." in err and err.split("]")[1].strip().split("(")[0] in r.stdout


def test_telecine_side_files_from_counts(exe, tmp_path):
    n = 43
    counts = np.zeros((n, 12), np.int32)
    counts[:, 2] = 40
    counts[:, 5] = 35
    film = []
    for c in range(2, n - 4, 5):                                   # combed pairs at frames c, c+1 (phase 2) ...
        if (c // 5) % 3 != 2:                                      # ... except every third cycle (video insert)
            counts[c, 2] = counts[c, 5] = 5000
            counts[c + 1, 2] = counts[c + 1, 5] = 4000
            film.append(c)
    cp = tmp_path / "c.bin"
    counts.tofile(cp)
    r = run(exe, "telecine", cp, n, 30000, 1001, tmp_path / "tc")
    assert ("film_cycles=%d" % len(film)) in r.stdout
    dur = [int(x) for x in open(tmp_path / "tc.duration.txt").read().split()]
    assert sum(dur) == n and len(dur) == n - len(film)
    # every film cycle is 1,1,2,1 with the long frame starting on the first combed frame
    starts = np.concatenate([[0], np.cumsum(dur)[:-1]])
    assert sorted(int(s) for s, d in zip(starts, dur) if d == 2) == film
    # the timecode file holds one stamp per output frame and the total; the reader recovers both
    out = run(exe, "timecode", tmp_path / "tc.timecode.txt").stdout.split()
    stamps = [float(x) for x in out[3:]]
    assert len(stamps) == len(dur) + 1
    assert stamps[-1] == pytest.approx(n * 1001 / 30.0, abs=1e-3)
    assert stamps[:-1] == [float(int(np.floor(s * 1001 / 30.0 + 0.5))) for s in starts]     # std::round: half away from zero
    # decimate accepts its own duration file
    assert run(exe, "decimate", tmp_path / "tc.duration.txt", n).stdout.startswith("frames=%d " % len(dur))


def _frame_result(n, elems):
    fr = np.zeros(n, np.int32)

    def fill(a, b, v):
        a = min(n, a)
        b = min(n, max(a, b))
        fr[a:b] = v
    for (sb, ss, se), (eb, es, ee) in elems:
        fill(ss, se + 1, 1)
        fill(se, es + 1, 2)
        fill(es + 1, ee + 1, 1)
    return fr


def test_eraselogo_fade_selection(exe, tmp_path):
    n, maxfade, rec, elems = ri.erase_fades_inputs()
    rp = tmp_path / "rec.bin"
    rec.tofile(rp)
    lg = synth.make_logo(32, 32, seed=2)
    lp = str(tmp_path / "logo.lgd")
    ab.Logo.create(lg["data"], 32, 32, 64, 32, 8, 0).save(lp, "t", 1)
    # without a logoframe file every frame goes through CalcFade2 (LogoScan.hpp:1263-1315)
    fp = tmp_path / "f0.bin"
    run(exe, "fades", lp, "-", rp, n, maxfade, fp)
    got = np.fromfile(fp, np.float32).reshape(n, 2)
    want = np.array([po.or_calc_fade2(rec, n, i) for i in range(n)], np.float32)
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
    # with one: frames whose +-maxfade/2 neighbourhood has a uniform state take 0 / 1 directly (:1317-1341)
    lf = tmp_path / "logof.txt"
    lf.write_text(ri.logoframe_file(elems))
    run(exe, "fades", lp, lf, rp, n, maxfade, fp)
    got = np.fromfile(fp, np.float32).reshape(n, 2)
    fr = _frame_result(n, elems)
    half = maxfade >> 1
    direct = 0
    for i in range(n):
        win = fr[np.clip(np.arange(i - half, i + half + 1), 0, n - 1)]
        if np.all(win == win[0]):
            exp = (1.0, 1.0) if fr[i] == 2 else (0.0, 0.0)
            direct += 1
        else:
            exp = po.or_calc_fade2(rec, n, i)
        assert tuple(np.float32(exp)) == tuple(got[i]), i
    assert 0 < direct < n
    # ... and so does the reference's OWN ReadLogoFrameFile + CalcFade (LogoScan.hpp:1317-1341,1421-1461; compiled from the
    # reference's lines into oracle/_ref, its results stored in tests/golden/ref_cases.json): the product's C++ driver picks
    # the same fades, frame for frame, bit for bit
    g = REF["erase_fades"]
    assert np.array_equal(np.array(g["state"], np.int32), fr)
    assert got.view(np.uint32).ravel().tolist() == g["logof_bits"]
    assert want.view(np.uint32).ravel().tolist() == g["no_logof_bits"]
    assert "Start and End must be cyclic" in g["cyclic_error"]
    if po.ref_available() and hasattr(po.ref_lib(), "ref_erase_fades"):
        rf, rstate = po.ref_erase_fades(rec, n, lf, maxfade)
        assert np.array_equal(rstate, fr)
        assert np.array_equal(rf.view(np.uint32), got.view(np.uint32))
        rf0, _ = po.ref_erase_fades(rec, n, None, maxfade)
        assert np.array_equal(rf0.view(np.uint32), want.view(np.uint32))
        lf.write_text("%6d S 0 ALL %6d %6d\n%6d S 0 ALL %6d %6d\n" % (22, 20, 26, 58, 55, 61))
        with pytest.raises(RuntimeError, match="Start and End must be cyclic"):
            po.ref_erase_fades(rec, n, lf, maxfade)
    # malformed files are rejected with the reference's message
    lf.write_text("%6d S 0 ALL %6d %6d\n%6d S 0 ALL %6d %6d\n" % (22, 20, 26, 58, 55, 61))
    r = run(exe, "fades", lp, lf, rp, n, maxfade, fp, ok=(4,))
    assert "Start and End must be cyclic" in r.stdout
    r = run(exe, "fades", tmp_path / "none.lgd", "-", rp, n, maxfade, fp, ok=(4,))
    assert "Failed to read logo file" in r.stdout


def test_filter_source_pass_loop(exe, tmp_path):
    """AMTFilterSource (FilteredSource.hpp:232-275,519-544): fresh environment per pass, AMT_* variables, AMT_PRE_PROC decides
    whether the pass is pulled and discarded, AMTDecimate appended when a duration file was left behind, timecodes read,
    AvisynthError converted to AviSynthException.  CPU-only source injected through the environment hook."""
    def run(script, n=23):
        d = tmp_path / script
        d.mkdir()
        r = subprocess.run([exe, "filterpass", str(d), str(n), script], capture_output=True, text=True, timeout=60)
        assert r.returncode == 0, r.stdout + r.stderr
        return r.stdout
    s = run("vfr")                      # Misc.cs:1305-1306: pre-process while AMT_PASS < 2
    assert "script: pass0(dev=3,tmp=" in s and "pass1(dev=3" in s and "pass2(dev=3" in s and "pass3" not in s
    assert "v0-0-0.avstmp" in s                                    # TranscodeSetting.hpp:875-880
    assert "preproc_passes=2" in s and "pulls=46" in s             # two passes x 23 frames pulled and discarded
    assert "out_frames=19" in s and "is_decimate=1" in s           # 23 source frames, four 2-frame durations -> 19
    assert "timecodes=20" in s and "vfrfps=60" in s                # 19 stamps + "# total:"; 60000/1001 grid fits best
    s = run("cfr")                      # Misc.cs:1311-1312: one pre-process pass
    assert "preproc_passes=1" in s and "pulls=23" in s and "pass2" not in s and "is_decimate=1" in s
    s = run("none")                     # no script: the source is the output, nothing is pulled
    assert "preproc_passes=0" in s and "pulls=0" in s and "out_frames=23" in s and "is_decimate=0" in s
    s = run("four")                     # at most four passes (FilteredSource.hpp:232)
    assert "script: pass0 pass1 pass2 pass3 \n" in s and "preproc_passes=4" in s and "pulls=92" in s
    s = run("throw")
    assert "AviSynthException: script failed in pass 0" in s      # :289-295


def test_source_frame_list_and_field_plan(exe):
    """StreamReform.hpp:874-904 (picture structure -> source frames) and AMTSource.hpp:524-551 (half-delay frames take their
    top field from the previous decoded picture; a repeated picture yields a second, undelayed frame)."""
    def run(pics):
        r = subprocess.run([exe, "fieldplan", pics], capture_output=True, text=True, timeout=30)
        assert r.returncode == 0
        return r.stdout.strip()
    # 0 FRAME, 3 TFF, 4 BFF, 6 BFF_RFF, 1 DOUBLING, 2 TRIPLING, 5 TFF_RFF
    assert run("0343663") == ("frames=9: 0/0,0@0.0 1/1,1@1.0 2h/1,2@1.5 3/3,3@3.0 4h/3,4@3.5 4/4,4@4.5 5h/4,5@5.5 5/5,5@6.5 6/6,6@8.0")
    assert run("125") == "frames=6: 0/0,0@0.0 0/0,0@1.0 1/1,1@2.0 1/1,1@3.0 1/1,1@4.0 2/2,2@5.0"
    # a delayed first picture has no predecessor: no frame is made for it and GetFrame serves the next cached one (:567-577)
    assert run("4412").startswith("frames=7: 0h/0,1@-0.5 1h/0,1@0.5 2/2,2@2.0 2/2,2@3.0")
