"""GPU parity tests: the CUDA path, called through the C ABI (ctypes), against the CPU oracle on the same bytes.
Bit-exact for the integer combing counters AND for the float logo scores (the kernels replicate the reference's
AVX summation tree and its sequential score sum); the 1e-5 relative tolerance of BASELINE.json is therefore not
needed and not used -- tests assert exact equality of the float bit patterns."""
import numpy as np
import pytest
import torch

import amatsukaze_b200 as ab
from amatsukaze_b200 import synth

pytestmark = pytest.mark.gpu

W, H = 256, 128
IMGX, IMGY = 160, 32


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def _logos(po, w=64, h=64, imgw=W, imgh=H, imgx=IMGX, imgy=IMGY, ratio=0.35):
    lg = synth.make_logo(w, h)
    p = ab.Logo.create(lg["data"], w, h, imgw, imgh, imgx, imgy)
    o = po.OracleLogo.create(lg["data"], w, h, imgw, imgh, imgx, imgy)
    P = {"raw": p, "deint": p.deint().create_mask(ratio), "top": p.field(0).create_mask(ratio), "bot": p.field(1).create_mask(ratio)}
    O = {"raw": o, "deint": o.deint().create_mask(ratio), "top": o.field(0).create_mask(ratio), "bot": o.field(1).create_mask(ratio)}
    return lg, P, O


def _clip(frames, w, h, on_device=True, bits=8):
    return ab.yv12_clip(frames, w, h, frames.shape[0], on_device, bits)


def test_scan_frames_bit_exact(ctx, oracle):
    po = oracle
    lg, P, O = _logos(po)
    n = 48
    fr = synth.make_frames(40, n, W, H, device="cuda", logo=lg, imgx=IMGX, imgy=IMGY, logo_period=40)
    out = ctx.scan_frames(_clip(fr, W, H), [P["deint"]]).cpu().numpy()
    Y, _, _ = synth.split_planes(fr, W, H)
    ref = np.stack([O["deint"].scan_frame(Y[i]) for i in range(n)])
    assert np.array_equal(_bits(out[:, 0, :]), _bits(ref))
    assert ref[:, 0].max() > 0.5 and ref[:, 0].min() < 0.1        # logo on and off both occur


def test_scan_frames_size_mismatch_and_multi_logo(ctx, oracle):
    po = oracle
    lg, P, O = _logos(po)
    lg2 = synth.make_logo(64, 64, seed=2)
    other = ab.Logo.create(lg2["data"], 64, 64, 1920, 1080, 100, 100).deint().create_mask(0.35)   # wrong frame size
    n = 5
    fr = synth.make_frames(60, n, W, H, device="cuda", logo=lg, imgx=IMGX, imgy=IMGY)
    out = ctx.scan_frames(_clip(fr, W, H), [other, P["deint"]]).cpu().numpy()
    assert np.all(out[:, 0, 0] == 0.0) and np.all(out[:, 0, 1] == -1.0)       # LogoScan.hpp:1551-1558
    Y, _, _ = synth.split_planes(fr, W, H)
    ref = np.stack([O["deint"].scan_frame(Y[i]) for i in range(n)])
    assert np.array_equal(_bits(out[:, 1, :]), _bits(ref))


def test_analyze_frames_bit_exact(ctx, oracle):
    po = oracle
    lg, P, O = _logos(po)
    n = 10
    fr = synth.make_frames(52, n, W, H, device="cuda", logo=lg, imgx=IMGX, imgy=IMGY, logo_period=20)
    out = ctx.analyze_frames(_clip(fr, W, H), P["deint"], P["top"], P["bot"]).cpu().numpy()
    Y, _, _ = synth.split_planes(fr, W, H)
    ref = np.stack([po.or_analyze_frame(O["deint"], O["top"], O["bot"], Y[i]) for i in range(n)])
    assert np.array_equal(_bits(out), _bits(ref))


def test_comb_bit_exact_small(ctx, oracle):
    po = oracle
    n = 9
    for (w, h, mode) in ((256, 128, "interlaced"), (224, 136, "telecine"), (352, 270, "interlaced"), (96, 36, "interlaced")):
        fr = synth.make_frames(0, n, w, h, device="cuda", mode=mode)
        prm = ab.default_comb_params()
        out = ctx.comb_frames(_clip(fr, w, h), prm).cpu().numpy()
        Y, U, V = synth.split_planes(fr, w, h)
        ref = po.or_comb_clip(Y, U, V, prm.as_list())
        assert np.array_equal(out, ref), (w, h, mode, out[:3], ref[:3])
        assert ref[:, 1].sum() > 0 and ref[:, 0].sum() > 0


def test_fused_and_host_path(ctx, oracle):
    po = oracle
    lg, P, O = _logos(po)
    n = 20
    fr = synth.make_frames(45, n, W, H, device="cuda", logo=lg, imgx=IMGX, imgy=IMGY, logo_period=30)
    prm = ab.default_comb_params()
    s, c = ctx.scan_comb_frames(_clip(fr, W, H), [P["deint"]], prm)
    Y, U, V = synth.split_planes(fr, W, H)
    rs = np.stack([O["deint"].scan_frame(Y[i]) for i in range(n)])
    rc = po.or_comb_clip(Y, U, V, prm.as_list())
    assert np.array_equal(_bits(s.cpu().numpy()[:, 0]), _bits(rs)) and np.array_equal(c.cpu().numpy(), rc)
    # same through HOST buffers (library stages frames through HBM itself)
    host = fr.cpu().numpy()
    s2, c2 = ctx.scan_comb_frames(_clip(host, W, H, on_device=False), [P["deint"]], prm)
    assert np.array_equal(_bits(s2[:, 0]), _bits(rs)) and np.array_equal(c2, rc)


# ----------------------------------------------------------------------------------------------------------------
# golden fixtures (produced by the reference's own code, tests/golden/gen_golden.py) through the C ABI
# ----------------------------------------------------------------------------------------------------------------
import json
import os

GOLD = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "logo_golden.json")))


def test_golden_scan_and_analyze(ctx):
    lg = synth.make_logo(64, 64, seed=1)
    fr = synth.make_frames(40, 24, W, H, seed=0x5EED0001, device="cuda", logo=lg, imgx=IMGX, imgy=IMGY, logo_period=20)
    raw = ab.Logo.create(lg["data"], 64, 64, W, H, IMGX, IMGY)
    de, top, bot = raw.deint().create_mask(0.35), raw.field(0).create_mask(0.35), raw.field(1).create_mask(0.35)
    clip = _clip(fr, W, H)
    out = ctx.scan_frames(clip, [de]).cpu().numpy()
    assert [_bits(out[i, 0]).tolist() for i in range(24)] == GOLD["scan_frame_bits"]
    an = ctx.analyze_frames(clip, de, top, bot).cpu().numpy()
    for k, i in enumerate(GOLD["analyze_frames"]):
        assert _bits(an[i]).tolist() == GOLD["analyze_bits"][k]
    de10 = raw.deint().create_mask(0.1)
    fades = (np.float32(0.1) * np.arange(20, dtype=np.float32)).astype(np.float32)       # LogoScan.hpp:967
    sweep = ctx.eval_fades(clip, de10, fades, frame0=12, nframes=1).cpu().numpy()
    assert _bits(sweep[0]).tolist() == GOLD["fade_sweep_bits"]


def test_scan_frames_16bit(ctx, oracle):
    """YUV420P10: maxv=1023, u16 samples; also the reference's byte-pitch quirk (LogoScan.hpp:1547,1561)."""
    po = oracle
    w, h, imgx, imgy = 256, 128, 96, 16
    lg, P, O = _logos(po, imgw=w, imgh=h, imgx=imgx, imgy=imgy)
    n = 6
    f8 = synth.make_frames(50, n, w, h, device="cuda", logo=lg, imgx=imgx, imgy=imgy, logo_period=20)
    f16 = (f8.to(torch.int32) * 4 + 1).to(torch.int16).contiguous()       # 10-bit range, packed like the 8-bit clip
    clip = ab.yv12_clip(f16, w, h, n, True, bits=10)
    out = ctx.scan_frames(clip, [P["deint"]]).cpu().numpy()
    Y16 = f16.cpu().numpy().view(np.uint16)[:, : w * h].reshape(n, h, w)
    ref = np.stack([O["deint"].scan_frame(Y16[i], maxv=1023.0) for i in range(n)])
    assert np.array_equal(_bits(out[:, 0]), _bits(ref))
    # quirk: element pitch = byte pitch (rows 2x apart); only legal while the doubled rows stay inside the plane
    with pytest.raises(ab.AmtkError, match="outside the frame"):
        ctx.scan_frames(clip, [P["deint"]], pitch_elems_override=2 * w)          # rows 2*(16..79) leave the plane
    lg0, P0, O0 = _logos(po, imgw=w, imgh=h, imgx=imgx, imgy=0)
    out_q = ctx.scan_frames(clip, [P0["deint"]], pitch_elems_override=2 * w).cpu().numpy()
    ref_q = np.stack([O0["deint"].scan_frame(Y16[i].reshape(h // 2, 2 * w), pitch=2 * w, maxv=1023.0) for i in range(n)])
    assert np.array_equal(_bits(out_q[:, 0]), _bits(ref_q))


def test_comb_thresholds_and_ragged_shapes(ctx, oracle):
    po = oracle
    prm = ab.default_comb_params()
    prm.th_move_y, prm.th_shima_y, prm.th_lshima_y = 1, 1, 2047
    prm.th_move_c, prm.th_shima_c, prm.th_lshima_c = 128, 700, 701
    for (w, h, n) in ((160, 34, 3), (128, 272, 5), (1952, 36, 2), (32, 1100, 2)):
        fr = synth.make_frames(3, n, w, h, device="cuda", mode="interlaced")
        out = ctx.comb_frames(_clip(fr, w, h), prm).cpu().numpy()
        Y, U, V = synth.split_planes(fr, w, h)
        assert np.array_equal(out, po.or_comb_clip(Y, U, V, prm.as_list())), (w, h)
    # extreme content: max-contrast alternating rows -> every pixel combs at the maximum response 1530
    w, h = 256, 128
    fr = torch.zeros((2, w * h * 3 // 2), dtype=torch.uint8, device="cuda")
    Yv = fr[:, : w * h].view(2, h, w)
    Yv[:, 0::2, :] = 255
    prm2 = ab.default_comb_params()
    prm2.th_shima_y, prm2.th_lshima_y = 1530, 1531
    out = ctx.comb_frames(_clip(fr, w, h), prm2).cpu().numpy()
    assert out[0, 1] + out[0, 4] == (h - 4) * w and out[0, 2] + out[0, 5] == 0 and out[:, 0].sum() == 0
    with pytest.raises(ab.AmtkError, match="th_move"):
        bad = ab.default_comb_params()
        bad.th_move_y = 0
        ctx.comb_frames(_clip(fr, w, h), bad)


def test_comb_range_sharding_and_chunked_host_path(ctx, oracle, monkeypatch):
    """Frame-range calls with a halo frame reproduce the whole-clip result (multi-GPU range sharding), and the
    host path stays exact when staging is forced into many small chunks."""
    po = oracle
    w, h, n = 352, 288, 23
    fr = synth.make_frames(0, n, w, h, device="cuda", mode="telecine")
    clip = _clip(fr, w, h)
    prm = ab.default_comb_params()
    whole = ctx.comb_frames(clip, prm).cpu().numpy()
    parts = np.concatenate([ctx.comb_frames(clip, prm, frame0=a, nframes=b - a).cpu().numpy() for a, b in ((0, 7), (7, 8), (8, 23))])
    assert np.array_equal(whole, parts)
    Y, U, V = synth.split_planes(fr, w, h)
    assert np.array_equal(whole, po.or_comb_clip(Y, U, V, prm.as_list()))
    # telecine: 2 of every 5 frames are combed -> their shima counts dominate
    sh = whole[:, 1] + whole[:, 4]
    assert sh[[2, 3]].min() > sh[[0, 1, 4]].max()
    monkeypatch.setenv("AMTK_STAGE_MB", "1")          # 1 MiB staging -> ~6 frames per chunk
    host = fr.cpu().numpy()
    lg, P, O = _logos(po, imgw=w, imgh=h, imgx=200, imgy=100)
    s, c = ctx.scan_comb_frames(_clip(host, w, h, on_device=False), [P["deint"]], prm)
    assert np.array_equal(c, whole)
    rs = np.stack([O["deint"].scan_frame(Y[i]) for i in range(n)])
    assert np.array_equal(_bits(s[:, 0]), _bits(rs))


def test_logoscan_accumulate_matches_oracle(ctx, oracle):
    po = oracle
    w, h, sx, sy, sw, sh = 320, 192, 200, 64, 64, 48
    n = 60
    lg = synth.make_logo(sw, sh, seed=4)
    fr = synth.make_frames(0, n, w, h, seed=0x5EED0004, device="cuda", mode="flat", logo=lg, imgx=sx, imgy=sy)
    clip = _clip(fr, w, h)
    acc = ctx.logo_scan(sw, sh, 12)
    valid = acc.add_frames(clip, sx, sy, 0, 40)
    valid2 = acc.add_frames(clip, sx, sy, 40, 20)            # accumulates across calls
    Y, U, V = synth.split_planes(fr, w, h)
    o = po.OracleScan(sw, sh, 12)
    ov = [o.add_frame(Y[i][sy:sy + sh, sx:sx + sw], U[i][sy // 2:(sy + sh) // 2, sx // 2:(sx + sw) // 2],
                      V[i][sy // 2:(sy + sh) // 2, sx // 2:(sx + sw) // 2]) for i in range(n)]
    assert np.concatenate([valid, valid2]).tolist() == ov and 0 < sum(ov) < n
    assert acc.num_valid == o.nframes
    assert np.array_equal(acc.sums(), o.sums())              # exact integers in doubles
    for clean in (False, True):
        a, b = acc.get_logo(255, clean), o.get_logo(255, clean)
        assert a is not None and np.array_equal(a.view(np.uint32), b.view(np.uint32))
    # frame_select (ReMakeLogo's minFades filter): only selected frames are offered
    acc2 = ctx.logo_scan(sw, sh, 12)
    sel = (np.arange(n) % 3 == 0).astype(np.uint8)
    v2 = acc2.add_frames(clip, sx, sy, select=sel)
    assert v2.tolist() == [a & int(b) for a, b in zip(ov, sel)]
    empty = ctx.logo_scan(sw, sh, 12)
    assert empty.get_logo(255) is None                       # "Insufficient logo frames"


def test_erase_logo_matches_oracle(ctx, oracle):
    po = oracle
    lg, P, O = _logos(po)
    n = 6
    fr = synth.make_frames(60, n, W, H, device="cuda", logo=lg, imgx=IMGX, imgy=IMGY)
    work = fr.clone()
    fades = np.array([[1.0, 1.0], [0.0, 0.0], [0.5, 0.5], [0.3, 0.7], [1.0, 0.0], [0.25, 0.25]], np.float32)
    ctx.erase_logo(_clip(work, W, H), P["raw"], fades)
    got = work.cpu().numpy()
    ref = fr.cpu().numpy().copy()
    for i in range(n):
        Y, U, V = [np.ascontiguousarray(p[i]) for p in synth.split_planes(ref, W, H)]
        po.or_erase_frame(O["raw"], Y, U, V, fades[i, 0], fades[i, 1])
        exp = np.concatenate([Y.ravel(), U.ravel(), V.ravel()])
        assert np.array_equal(got[i], exp), i
    assert np.array_equal(got[1], fr.cpu().numpy()[1])       # fade 0 leaves the frame untouched
    assert not np.array_equal(got[0], fr.cpu().numpy()[0])


@pytest.mark.timeout(600)
def test_full_size_properties_1080p(ctx, oracle):
    """BASELINE-size frames (1920x1080): spot parity on a few frames + size-independent properties."""
    po = oracle
    w, h, n, imgx, imgy = 1920, 1080, 40, 1700, 60
    lg = synth.make_logo(64, 64)
    fr = torch.empty((n, w * h * 3 // 2), dtype=torch.uint8, device="cuda")
    for n0 in range(0, n, 10):
        synth.make_frames(100 + n0, 10, w, h, device="cuda", logo=lg, imgx=imgx, imgy=imgy, logo_period=30, out=fr[n0:n0 + 10])
    clip = _clip(fr, w, h)
    logo = ab.Logo.create(lg["data"], 64, 64, w, h, imgx, imgy).deint().create_mask(0.35)
    prm = ab.default_comb_params()
    s, c = ctx.scan_comb_frames(clip, [logo], prm)
    s, c = s.cpu().numpy(), c.cpu().numpy()
    o = po.OracleLogo.create(lg["data"], 64, 64, w, h, imgx, imgy).deint().create_mask(0.35)
    Y, U, V = synth.split_planes(fr, w, h)
    for i in (0, 1, 17, 39):
        assert np.array_equal(_bits(s[i, 0]), _bits(o.scan_frame(Y[i])))
        j = max(i - 1, 0)
        assert np.array_equal(c[i], po.or_comb_frame((Y[i], U[i], V[i]), (Y[j], U[j], V[j]), prm.as_list()))
    # properties: counters bounded by the number of pixels of their field; lshima <= shima; frame 0 has no motion
    top_y = (h // 2) * w
    assert (c[:, [0, 1, 2, 3, 4, 5]] <= top_y).all() and (c[:, 2] <= c[:, 1]).all() and (c[:, 5] <= c[:, 4]).all()
    assert c[0, [0, 3, 6, 9]].sum() == 0
    # split / merge invariance (range sharding with halo) and determinism
    a = ctx.comb_frames(clip, prm, 0, 13).cpu().numpy()
    b = ctx.comb_frames(clip, prm, 13, 27).cpu().numpy()
    assert np.array_equal(np.concatenate([a, b]), c)
    s2, c2 = ctx.scan_comb_frames(clip, [logo], prm)
    assert np.array_equal(s2.cpu().numpy().view(np.uint32), s.view(np.uint32)) and np.array_equal(c2.cpu().numpy(), c)
    assert s[:, 0, 0].max() > 0.8 and s[:, 0, 0].min() < 0.2


def test_scan_frames_unaligned_pitch_fallback(ctx, oracle):
    """Row pitch not a multiple of 16 bytes: TMA cannot describe the plane, the kernel falls back to plain loads."""
    po = oracle
    w, h, imgx, imgy = 200, 96, 120, 20
    lg = synth.make_logo(48, 40, seed=6)
    p = ab.Logo.create(lg["data"], 48, 40, w, h, imgx, imgy).deint().create_mask(0.35)
    o = po.OracleLogo.create(lg["data"], 48, 40, w, h, imgx, imgy).deint().create_mask(0.35)
    n = 7
    fr = synth.make_frames(20, n, w, h, device="cuda", logo=lg, imgx=imgx, imgy=imgy, logo_period=10)
    out = ctx.scan_frames(_clip(fr, w, h), [p]).cpu().numpy()
    Y, _, _ = synth.split_planes(fr, w, h)
    ref = np.stack([o.scan_frame(Y[i]) for i in range(n)])
    assert np.array_equal(_bits(out[:, 0]), _bits(ref))
    # the combing metric takes the generic (non-TMA) kernel for this layout: same counters
    got = ctx.comb_frames(_clip(fr, w, h)).cpu().numpy()
    _, U, V = synth.split_planes(fr, w, h)
    assert np.array_equal(got, po.or_comb_clip(Y, U, V, ab.default_comb_params().as_list()))


def test_comb_16bit(ctx, oracle, monkeypatch):
    """YUV420P10 clips: the integer spec on u16 samples -- streaming (TMA, fp32 stencil) kernel incl. the merged U|V
    remainder tile and range calls with a halo frame, and the generic kernel on the same data."""
    po = oracle
    prm = ab.default_comb_params()
    prm.th_move_y, prm.th_shima_y, prm.th_lshima_y = 80, 48, 3000
    prm.th_move_c, prm.th_shima_c, prm.th_lshima_c = 200, 64, 144
    for (w, h, n) in ((224, 136, 7), (320, 150, 5)):
        f8 = synth.make_frames(2, n, w, h, device="cuda", mode="telecine")
        f16 = (f8.to(torch.int32) * 4 + (f8.to(torch.int32) & 3)).to(torch.int16).contiguous()
        clip = ab.yv12_clip(f16, w, h, n, True, bits=10)
        got = ctx.comb_frames(clip, prm).cpu().numpy()
        a16 = f16.cpu().numpy().view(np.uint16)
        ysz, csz = w * h, (w // 2) * (h // 2)
        Y = a16[:, :ysz].reshape(n, h, w); U = a16[:, ysz:ysz + csz].reshape(n, h // 2, w // 2); V = a16[:, ysz + csz:].reshape(n, h // 2, w // 2)
        ref = po.or_comb_clip(Y, U, V, prm.as_list())
        assert np.array_equal(got, ref) and ref[:, 1].sum() > 0, (w, h)
        part = np.concatenate([ctx.comb_frames(clip, prm, 0, 3).cpu().numpy(), ctx.comb_frames(clip, prm, 3, n - 3).cpu().numpy()])
        assert np.array_equal(part, ref)
        monkeypatch.setenv("AMTK_COMB_GENERIC", "1")
        g = ab.Context(0, torch.cuda.current_stream().cuda_stream)
        monkeypatch.delenv("AMTK_COMB_GENERIC")
        try:
            assert np.array_equal(g.comb_frames(clip, prm).cpu().numpy(), ref)
        finally:
            g.close()
            ab.Context(0, torch.cuda.current_stream().cuda_stream).close()      # restores the default knobs
    # full-range 16-bit samples and the largest move threshold
    w, h, n = 256, 136, 3
    rnd = torch.randint(0, 65536, (n, w * h * 3 // 2), device="cuda", dtype=torch.int32).to(torch.int16).contiguous()
    clip = ab.yv12_clip(rnd, w, h, n, True, bits=16)
    prm.th_move_y, prm.th_move_c, prm.th_shima_y, prm.th_lshima_y = 32768, 1, 100000, 300000
    got = ctx.comb_frames(clip, prm).cpu().numpy()
    a16 = rnd.cpu().numpy().view(np.uint16)
    ysz, csz = w * h, (w // 2) * (h // 2)
    ref = po.or_comb_clip(a16[:, :ysz].reshape(n, h, w), a16[:, ysz:ysz + csz].reshape(n, h // 2, w // 2),
                          a16[:, ysz + csz:].reshape(n, h // 2, w // 2), prm.as_list())
    assert np.array_equal(got, ref)


def test_scan_logo_pipeline(ctx, oracle, tmp_path):
    """amtk_scan_logo = the reference's ScanLogo pipeline (LogoScan.hpp:1058-1098): MakeInitialLogo, ReMakeLogo x2,
    Save -- compared with the same pipeline composed from the oracle's pieces."""
    po = oracle
    w, h, sx, sy, sw, sh, n, thy, maxf = 320, 192, 200, 64, 64, 48, 90, 12, 40
    lg = synth.make_logo(sw, sh, seed=4)
    fr = synth.make_frames(0, n, w, h, seed=0x5EED0004, device="cuda", mode="flat", logo=lg, imgx=sx, imgy=sy)
    clip = _clip(fr, w, h)
    dst = str(tmp_path / "gen.lgd")
    calls = []
    ctx.scan_logo(clip, dst, sx, sy, sw, sh, thy, maxf, service_id=410, cb=lambda p, a, b, c: calls.append((p, a, b, c)) or True)
    # callback contract of the reference (LogoScan.hpp:905-910,977-982,1071): every 200 frames read in MakeInitialLogo (none
    # here: the limit is hit after < 200 frames), every 100 stored frames in each ReMakeLogo (i = 0 only), then (1, n, n, n)
    assert calls == [(50.0, 0, maxf, maxf), (75.0, 0, maxf, maxf), (1.0, maxf, maxf, maxf)], calls
    got = ab.Logo.load(dst)
    gi = got.info()
    assert (gi.w, gi.h, gi.imgw, gi.imgh, gi.imgx, gi.imgy) == (sw, sh, w, h, sx, sy)
    # ---- oracle composition ----
    Y, U, V = synth.split_planes(fr, w, h)
    roi = lambda i: (Y[i][sy:sy + sh, sx:sx + sw], U[i][sy // 2:(sy + sh) // 2, sx // 2:(sx + sw) // 2], V[i][sy // 2:(sy + sh) // 2, sx // 2:(sx + sw) // 2])
    sc = po.OracleScan(sw, sh, thy)
    stored = []
    for i in range(n):
        if len(stored) >= maxf:
            break
        if sc.add_frame(*roi(i)):
            stored.append(i)
    assert len(stored) == maxf and stored[-1] < n - 10        # the cut-off really bites
    data = sc.get_logo(255, False)
    for _ in range(2):
        de = po.OracleLogo.create(data, sw, sh, sw, sh, 0, 0).deint().create_mask(0.1)
        keep = []
        for i in stored:
            ry = np.ascontiguousarray(roi(i)[0])
            dd = np.zeros(sw * sh + 8, np.float32)
            po.oracle_lib().amtk_or_deint_y_u8(dd.ctypes.data_as(po.c_float_p), ry.ctypes.data_as(po.c_u8_p), sw, sw, sh)
            res = [abs(np.float32(de.evaluate(dd, 255.0, np.float32(0.1) * np.float32(fi)))) for fi in range(20)]
            if int(np.argmin(res)) > 8:
                keep.append(i)
        assert 0 < len(keep) < len(stored)
        sc2 = po.OracleScan(sw, sh, thy)
        for i in keep:
            sc2.add_frame(*roi(i))
        data = sc2.get_logo(255, True)
        assert data is not None
    assert np.array_equal(got.tables()["data"].view(np.uint32), data.view(np.uint32))
    # a longer clip: the 200-frame and 100-frame callback cadences, progress formulas and a cancel in the MIDDLE of a pass
    n2 = 450
    fr2 = synth.make_frames(0, n2, w, h, seed=0x5EED0005, device="cuda", mode="flat", logo=lg, imgx=sx, imgy=sy)
    clip2 = _clip(fr2, w, h)
    calls2 = []
    ctx.scan_logo(clip2, dst, sx, sy, sw, sh, thy, 100000, cb=lambda p, a, b, c: calls2.append((p, a, b, c)) or True)
    Y2, U2, V2 = synth.split_planes(fr2, w, h)
    sc3 = po.OracleScan(sw, sh, thy)
    nv = [0]
    for i in range(n2):
        nv.append(nv[-1] + (1 if sc3.add_frame(Y2[i][sy:sy + sh, sx:sx + sw], U2[i][sy // 2:(sy + sh) // 2, sx // 2:(sx + sw) // 2],
                                               V2[i][sy // 2:(sy + sh) // 2, sx // 2:(sx + sw) // 2]) else 0))
    nvalid = nv[-1]
    assert nvalid > 200
    want = [(np.float32(50.0 * r / n2), r, 0, nv[r]) for r in (200, 400)]
    for base in (50.0, 75.0):
        want += [(np.float32(np.float32(i) / np.float32(nvalid) * np.float32(25.0) + np.float32(base)), i, nvalid, nvalid) for i in range(0, nvalid, 100)]
    want.append((1.0, nvalid, nvalid, nvalid))
    assert [(np.float32(c[0]),) + c[1:] for c in calls2] == [(np.float32(x[0]),) + x[1:] for x in want], (calls2, want)
    seen = []
    with pytest.raises(ab.AmtkError, match="Cancel requested"):
        ctx.scan_logo(clip2, dst, sx, sy, sw, sh, thy, 100000, cb=lambda p, a, b, c: seen.append(a) or len(seen) < 5)
    assert len(seen) == 5                                    # stopped inside the first ReMakeLogo, not after it
    # cancel + insufficient frames behave like the reference
    with pytest.raises(ab.AmtkError, match="Cancel requested"):
        ctx.scan_logo(clip, dst, sx, sy, sw, sh, thy, maxf, cb=lambda *a: False)
    with pytest.raises(ab.AmtkError, match="Insufficient logo frames"):
        ctx.scan_logo(clip, dst, sx, sy, sw, sh, 0, maxf)


def test_weave_frames_matches_mergefield(ctx):
    """AMTSource::MergeField/Copy1/Copy2 (AMTSource.hpp:291-355): even rows from `top`, odd rows from `bottom`,
    planar and NV12 sources, 8- and 16-bit."""
    import ref_inputs as ri
    w, h, n, top, bot = ri.WEAVE
    src8 = ri.weave_frames("cuda")
    top = np.array(top, np.int32)
    bot = np.array(bot, np.int32)                         # half-delay: bottom field of the next decoded frame
    for bits in (8, 10):
        src = src8 if bits == 8 else (src8.to(torch.int32) * 4 + 2).to(torch.int16).contiguous()
        dst = torch.zeros_like(src)
        ctx.weave_frames(ab.yv12_clip(src, w, h, n, True, bits), ab.yv12_clip(dst, w, h, n, True, bits), top, bot)
        a = src.cpu().numpy(); a = a if bits == 8 else a.view(np.uint16)
        g = dst.cpu().numpy(); g = g if bits == 8 else g.view(np.uint16)
        ysz, csz = w * h, (w // 2) * (h // 2)
        for k in range(n):
            for (o, rows, cols) in ((0, h, w), (ysz, h // 2, w // 2), (ysz + csz, h // 2, w // 2)):
                t = a[top[k], o:o + rows * cols].reshape(rows, cols)
                b = a[bot[k], o:o + rows * cols].reshape(rows, cols)
                exp = t.copy(); exp[1::2] = b[1::2]
                assert np.array_equal(g[k, o:o + rows * cols].reshape(rows, cols), exp), (bits, k, o)
    # NV12 source: interleaved UV plane split into U and V
    ysz, csz = w * h, (w // 2) * (h // 2)
    a = src8.cpu().numpy()
    nv = a.copy()
    uv = np.stack([a[:, ysz:ysz + csz], a[:, ysz + csz:]], axis=2).reshape(n, 2 * csz)
    nv[:, ysz:] = uv
    nv_t = torch.from_numpy(nv).cuda()
    sclip = ab.yv12_clip(nv_t, w, h, n, True)
    sclip.pitch_uv = w                                     # interleaved UV rows are `width` bytes long
    dst = torch.zeros_like(src8)
    ctx.weave_frames(sclip, ab.yv12_clip(dst, w, h, n, True), top, bot, src_is_nv12=True)
    ref = torch.zeros_like(src8)
    ctx.weave_frames(ab.yv12_clip(src8, w, h, n, True), ab.yv12_clip(ref, w, h, n, True), top, bot)
    assert torch.equal(dst, ref)
    # ... and both equal the reference's OWN MergeField / Copy1 / Copy2 (AMTSource.hpp:291-355; its outputs stored as digests
    # in tests/golden/ref_cases.json, and computed live where oracle/_ref is built)
    import hashlib
    from oracle import pyoracle as po
    gw = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "ref_cases.json")))["weave"]
    g = dst.cpu().numpy()
    for k in range(n):
        sha = hashlib.sha256(np.ascontiguousarray(g[k]).tobytes()).hexdigest()
        assert sha == gw["planar_sha"][k] and sha == gw["nv12_sha"][k], k
    if po.ref_has_mergefield():
        for k in range(n):
            assert np.array_equal(g[k], po.ref_merge_field(a[top[k]], a[bot[k]], w, h)), ("planar", k)
            assert np.array_equal(g[k], po.ref_merge_field(nv[top[k]], nv[bot[k]], w, h, nv12=True)), ("nv12", k)
    with pytest.raises(ab.AmtkError, match="index outside"):
        ctx.weave_frames(ab.yv12_clip(src8, w, h, n, True), ab.yv12_clip(dst, w, h, n, True), top, bot + 1)


def test_logo_sizes_small_large_multislice(ctx, oracle):
    """Logo geometry sweep: PXT=1 (few features), several pixel slices (> 1536 features), A/B-through-L1 and
    one-fade-per-pass shared-memory plans for large logos; also the analyze path on a wide flat logo."""
    po = oracle
    W2, H2 = 640, 288
    n = 3
    fr = synth.make_frames(11, n, W2, H2, device="cuda", mode="interlaced")
    Y, _, _ = synth.split_planes(fr, W2, H2)
    for (w, h, ratio, imgx, imgy) in ((32, 32, 0.35, 300, 100), (128, 96, 0.35, 410, 66), (200, 112, 0.2, 96, 120), (256, 90, 0.5, 320, 4)):
        lg = synth.make_logo(w, h, seed=w)
        p = ab.Logo.create(lg["data"], w, h, W2, H2, imgx, imgy)
        o = po.OracleLogo.create(lg["data"], w, h, W2, H2, imgx, imgy)
        pd, od = p.deint().create_mask(ratio), o.deint().create_mask(ratio)
        assert pd.info().count == od.s.count
        out = ctx.scan_frames(_clip(fr, W2, H2), [pd]).cpu().numpy()
        ref = np.stack([od.scan_frame(Y[i]) for i in range(n)])
        assert np.array_equal(_bits(out[:, 0]), _bits(ref)), (w, h, pd.info().count)
        if h % 2 == 0 and h // 2 >= 5:
            pt, pb = p.field(0).create_mask(ratio), p.field(1).create_mask(ratio)
            ot, ob = o.field(0).create_mask(ratio), o.field(1).create_mask(ratio)
            an = ctx.analyze_frames(_clip(fr, W2, H2), pd, pt, pb, nframes=2).cpu().numpy()
            ra = np.stack([po.or_analyze_frame(od, ot, ob, Y[i]) for i in range(2)])
            assert np.array_equal(_bits(an), _bits(ra)), (w, h)
    huge = synth.make_logo(256, 128, seed=9)
    ph = ab.Logo.create(huge["data"], 256, 128, W2, H2, 64, 32).deint().create_mask(0.1)
    with pytest.raises(ab.AmtkError, match="too large"):
        ctx.scan_frames(_clip(fr, W2, H2), [ph])


def test_empty_single_and_bad_ranges(ctx, oracle):
    po = oracle
    lg, P, O = _logos(po)
    fr = synth.make_frames(77, 3, W, H, device="cuda", logo=lg, imgx=IMGX, imgy=IMGY)
    clip = _clip(fr, W, H)
    prm = ab.default_comb_params()
    # empty range: succeeds, returns empty arrays
    assert ctx.comb_frames(clip, prm, 1, 0).shape[0] == 0
    assert ctx.scan_frames(clip, [P["deint"]], 2, 0).shape[0] == 0
    # single frame in the middle: move compares with the real predecessor
    one = ctx.comb_frames(clip, prm, 2, 1).cpu().numpy()
    Y, U, V = synth.split_planes(fr, W, H)
    assert np.array_equal(one[0], po.or_comb_frame((Y[2], U[2], V[2]), (Y[1], U[1], V[1]), prm.as_list()))
    # a one-frame clip: prev(0) = itself -> no motion
    c1 = _clip(fr[:1].contiguous(), W, H)
    s, c = ctx.scan_comb_frames(c1, [P["deint"]], prm)
    assert c.cpu().numpy()[0, [0, 3, 6, 9]].sum() == 0
    assert np.array_equal(_bits(s.cpu().numpy()[0, 0]), _bits(O["deint"].scan_frame(Y[0])))
    for (f0, n) in ((-1, 2), (2, 2), (0, 4)):
        with pytest.raises(ab.AmtkError, match="frame range"):
            ctx.comb_frames(clip, prm, f0, n)
    with pytest.raises(ab.AmtkError, match="no mask"):
        ctx.scan_frames(clip, [P["raw"].deint()])
