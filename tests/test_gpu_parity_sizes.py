"""GPU parity at BASELINE.json's own sizes (VERDICT r1, next-round item 1c): configs[2] geometry (1440x1080: 11.25 luma
tiles, a quarter-used last tile column, 5.625 chroma tiles), 8- and 10-bit, against the spec oracle; configs[3]
(LogoScan accumulation over 10000 1920x1080 frames, ROI 64x64 and 256x128) against the reference's own LogoScan code
(oracle/_ref) where it exists, else the C port; a whole 1080p clip against the reference-compiled logo code.  Everything
goes through the C ABI."""
import hashlib
import json
import os

import numpy as np
import pytest
import torch

import amatsukaze_b200 as ab
import ref_inputs as ri
from amatsukaze_b200 import synth

pytestmark = pytest.mark.gpu
# the reference's own results at these sizes (tests/golden/gen_golden.py --sizes): the comparison with the reference holds
# where oracle/_ref is not built
REF = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "ref_sizes.json")))


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def _digest(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def _gen(n0, n, w, h, **kw):
    return ri.gen_frames(n0, n, w, h, "cuda", **kw)


@pytest.mark.timeout(900)
def test_comb_1440x1080_8bit_and_10bit(ctx, oracle):
    po = oracle
    w, h, n = 1440, 1080, 18
    prm = ab.default_comb_params()
    f8 = _gen(3, n, w, h, mode="telecine")
    got = ctx.comb_frames(ab.yv12_clip(f8, w, h, n, True), prm).cpu().numpy()
    Y, U, V = synth.split_planes(f8, w, h)
    ref = np.stack([po.or_comb_frame((Y[i], U[i], V[i]), (Y[max(i - 1, 0)], U[max(i - 1, 0)], V[max(i - 1, 0)]), prm.as_list(), "avx2")
                    for i in range(n)])
    assert np.array_equal(got, ref), np.argwhere(got != ref)[:5]
    # the scalar normative form on a few frames (AVX2 == scalar is a CPU test; this is the direct witness)
    for i in (0, 1, 9, 17):
        j = max(i - 1, 0)
        assert np.array_equal(got[i], po.or_comb_frame((Y[i], U[i], V[i]), (Y[j], U[j], V[j]), prm.as_list()))
    assert ref[:, [1, 4]].sum() > 0 and ref[1:, 0].sum() > 0
    # range calls with a halo frame give the same rows
    part = np.concatenate([ctx.comb_frames(ab.yv12_clip(f8, w, h, n, True), prm, 0, 7).cpu().numpy(),
                           ctx.comb_frames(ab.yv12_clip(f8, w, h, n, True), prm, 7, n - 7).cpu().numpy()])
    assert np.array_equal(part, ref)
    # YUV420P10: same geometry, 16-bit samples (fp32 stencil path)
    n10 = 16
    f16 = (f8[:n10].to(torch.int32) * 4 + (f8[:n10].to(torch.int32) & 3)).to(torch.int16).contiguous()
    p10 = ab.default_comb_params()
    p10.th_move_y, p10.th_shima_y, p10.th_lshima_y = 80, 48, 144
    p10.th_move_c, p10.th_shima_c, p10.th_lshima_c = 96, 64, 192
    got10 = ctx.comb_frames(ab.yv12_clip(f16, w, h, n10, True, bits=10), p10).cpu().numpy()
    a16 = f16.cpu().numpy().view(np.uint16)
    ysz, csz = w * h, (w // 2) * (h // 2)
    Y = a16[:, :ysz].reshape(n10, h, w); U = a16[:, ysz:ysz + csz].reshape(n10, h // 2, w // 2); V = a16[:, ysz + csz:].reshape(n10, h // 2, w // 2)
    ref10 = po.or_comb_clip(Y, U, V, p10.as_list())
    assert np.array_equal(got10, ref10) and ref10[:, 1].sum() > 0


@pytest.mark.timeout(900)
def test_scan_and_analyze_1440x1080(ctx, oracle):
    """configs[0]'s geometry (1440x1080, 64x64 template at (1280, 64)) on the GPU, against the reference's own code."""
    po = oracle
    w, h, n, imgx, imgy = ri.SCAN_1440
    lg = synth.make_logo(64, 64)
    fr = ri.scan_1440_frames(lg, "cuda")
    raw = ab.Logo.create(lg["data"], 64, 64, w, h, imgx, imgy)
    de, top, bot = raw.deint().create_mask(0.35), raw.field(0).create_mask(0.35), raw.field(1).create_mask(0.35)
    clip = ab.yv12_clip(fr, w, h, n, True)
    s = ctx.scan_frames(clip, [de]).cpu().numpy()
    a = ctx.analyze_frames(clip, de, top, bot).cpu().numpy()
    Y, _, _ = synth.split_planes(fr, w, h)
    if po.ref_available():
        r = po.RefLogo.create(lg["data"], 64, 64, w, h, imgx, imgy)
        rde, rtop, rbot = r.deint().create_mask(0.35), r.field(0).create_mask(0.35), r.field(1).create_mask(0.35)
        rs = np.stack([po.ref_scan_frame(rde, Y[i]) for i in range(n)])
        ra = np.stack([po.ref_analyze_frame(rde, rtop, rbot, Y[i]) for i in range(0, n, 5)])
    else:
        o = po.OracleLogo.create(lg["data"], 64, 64, w, h, imgx, imgy)
        ode, otop, obot = o.deint().create_mask(0.35), o.field(0).create_mask(0.35), o.field(1).create_mask(0.35)
        rs = np.stack([ode.scan_frame(Y[i]) for i in range(n)])
        ra = np.stack([po.or_analyze_frame(ode, otop, obot, Y[i]) for i in range(0, n, 5)])
    assert np.array_equal(_bits(s[:, 0]), _bits(rs))
    assert np.array_equal(_bits(a[0:n:5]), _bits(ra))
    assert rs[:, 0].max() > 0.5 and rs[:, 0].min() < 0.2
    g = REF["scan_analyze_1440"]
    assert _bits(s[:, 0]).ravel().tolist() == g["scan_bits"]
    assert g["analyze_frames"] == list(range(0, n, 5)) and _bits(a[0:n:5]).ravel().tolist() == g["analyze_bits"]


@pytest.mark.timeout(1800)
def test_logoscan_10000_frames_1080p(ctx, oracle):
    """configs[3]: 10000 resident 1920x1080 frames (31 GB), ROI 64x64 and 256x128: u64 sums, gridDim.y frame splits,
    validity per frame, and the derived logo (A/B planes) -- all exact."""
    po = oracle
    w, h, n = ri.LOGOSCAN_10K
    free, _ = torch.cuda.mem_get_info()
    if free < 36 * (1 << 30):
        pytest.skip("needs 36 GB of free HBM")
    lg = synth.make_logo(64, 64)
    fr = torch.empty((n, w * h * 3 // 2), dtype=torch.uint8, device="cuda")
    for k in range(0, n, 20):
        ri.logoscan_10k_frames(k, 20, lg, "cuda", out=fr[k:k + 20])
    clip = ab.yv12_clip(fr, w, h, n, True)
    ysz, csz = w * h, (w // 2) * (h // 2)
    for (sx, sy, sw, sh) in ri.LOGOSCAN_10K_ROIS:
        acc = ctx.logo_scan(sw, sh, 12)
        valid = acc.add_frames(clip, sx, sy, 0, 6000)
        valid = np.concatenate([valid, acc.add_frames(clip, sx, sy, 6000, 4000)])        # accumulates across calls
        # ROI stacks to the host (full frames would be 31 GB): exactly the bytes LogoScan::AddFrame reads
        Yr = fr[:, :ysz].view(n, h, w)[:, sy:sy + sh, sx:sx + sw].contiguous().cpu().numpy()
        Ur = fr[:, ysz:ysz + csz].view(n, h // 2, w // 2)[:, sy // 2:(sy + sh) // 2, sx // 2:(sx + sw) // 2].contiguous().cpu().numpy()
        Vr = fr[:, ysz + csz:].view(n, h // 2, w // 2)[:, sy // 2:(sy + sh) // 2, sx // 2:(sx + sw) // 2].contiguous().cpu().numpy()
        o = po.RefScan(sw, sh, 12) if po.ref_available() else po.OracleScan(sw, sh, 12)
        ov = np.array([o.add_frame(Yr[i], Ur[i], Vr[i]) for i in range(n)], np.uint8)
        assert np.array_equal(valid, ov), (sw, sh, int((valid != ov).sum()))
        assert 0 < int(ov.sum()) < n and acc.num_valid == o.nframes == int(ov.sum())
        assert np.array_equal(acc.sums(), o.sums())              # exact integers (< 2^53) in doubles
        g = REF["logoscan_10k"]["%dx%d" % (sw, sh)]
        assert _digest(valid.astype(np.uint8)) == g["valid_sha"] and acc.num_valid == g["nframes"]
        assert _digest(acc.sums()) == g["sums_sha"]
        for clean in (False, True):
            a, b = acc.get_logo(255, clean), o.get_logo(255, clean)
            assert a is not None and b is not None and np.array_equal(a.view(np.uint32), b.view(np.uint32))
            assert _digest(a) == g["logo_clean_sha" if clean else "logo_sha"]
        del acc


@pytest.mark.timeout(900)
def test_whole_clip_1080p_against_reference_code(ctx, oracle):
    """1000 consecutive 1080p frames of the bench clip (enough for all three tiers of the streaming kernel's work queue:
    32-, 8- and 4-frame items): every logo score bit-identical with the reference's own compiled code, every combing
    counter identical with the spec (AVX2 form; scalar form on a subset)."""
    po = oracle
    w, h, n, imgx, imgy = ri.WHOLE_CLIP
    lg = synth.make_logo(64, 64)
    fr = ri.whole_clip_frames(lg, "cuda")
    logo = ab.Logo.create(lg["data"], 64, 64, w, h, imgx, imgy).deint().create_mask(0.35)
    prm = ab.default_comb_params()
    s, c = ctx.scan_comb_frames(ab.yv12_clip(fr, w, h, n, True), [logo], prm)
    s, c = s.cpu().numpy(), c.cpu().numpy()
    host = fr.cpu().numpy()
    b = po.CpuBench(w, h, lg["data"], imgx, imgy, po.usable_cpu_threads(), 0.35)
    _, rs, rc = b.run(host, prm.as_list(), 3, "avx2")
    _, _, rc_s = b.run(host[:24], prm.as_list(), 2, "scalar")
    b.close()
    assert np.array_equal(_bits(s[:, 0]), _bits(rs))
    assert _digest(_bits(s[:, 0])) == REF["whole_clip_1080p"]["scores_sha"] and REF["whole_clip_1080p"]["frames"] == n
    assert np.array_equal(c, rc) and np.array_equal(c[:24], rc_s)
    # host-buffer path over the same clip (staged through HBM by the library): identical
    s2, c2 = ctx.scan_comb_frames(ab.yv12_clip(host, w, h, n, False), [logo], prm)
    assert np.array_equal(_bits(s2[:, 0]), _bits(rs)) and np.array_equal(c2, rc)


def test_logo_outlives_its_context(native_lib):
    """ADVICE r1 (medium): a logo only remembers the device ordinal, so closing the context that first evaluated it and
    destroying / re-using the logo afterwards is legal."""
    w, h = 256, 128
    lg = synth.make_logo(64, 64)
    fr = synth.make_frames(40, 4, w, h, device="cuda", logo=lg, imgx=160, imgy=32)
    clip = ab.yv12_clip(fr, w, h, 4, True)
    logo = ab.Logo.create(lg["data"], 64, 64, w, h, 160, 32).deint().create_mask(0.35)
    c1 = ab.Context(0, torch.cuda.current_stream().cuda_stream)
    a = c1.scan_frames(clip, [logo]).cpu().numpy()
    c1.close()
    c2 = ab.Context(0, torch.cuda.current_stream().cuda_stream)        # a second context may evaluate the same logo
    b = c2.scan_frames(clip, [logo]).cpu().numpy()
    c2.close()
    assert np.array_equal(_bits(a), _bits(b))
    del logo                                                            # destroyed after both contexts are gone
    torch.cuda.synchronize()


@pytest.mark.parametrize("bits", [8, 10])
def test_host_clips_upload_only_the_roi(ctx, oracle, bits):
    """Host-buffer calls of the logo entry points move only the logo / scan rectangle over PCIe (VERDICT r1 weak #6) and
    return exactly what the device-resident call returns -- odd alignments included (imgx not a multiple of 16 or 32)."""
    w, h, n = 416, 240, 23
    for (imgx, imgy, lw, lh) in ((150, 34, 64, 48), (20, 0, 70, 40), (416 - 64, 240 - 64, 64, 64), (2, 190, 48, 50)):
        lg = synth.make_logo(lw, lh, seed=3)
        f8 = synth.make_frames(11, n, w, h, device="cuda", logo=lg, imgx=imgx, imgy=imgy, logo_period=12)
        if bits == 8:
            fr = f8
        else:
            fr = (f8.to(torch.int32) * 4 + (f8.to(torch.int32) & 3)).to(torch.int16).contiguous()
        raw = ab.Logo.create(lg["data"], lw, lh, w, h, imgx, imgy)
        de, top, bot = raw.deint().create_mask(0.35), raw.field(0).create_mask(0.35), raw.field(1).create_mask(0.35)
        dclip = ab.yv12_clip(fr, w, h, n, True, bits)
        host = fr.cpu().numpy()
        hclip = ab.yv12_clip(host, w, h, n, False, bits)
        full = host.nbytes
        s_dev = ctx.scan_frames(dclip, [de]).cpu().numpy()
        s_host = ctx.scan_frames(hclip, [de])
        assert np.array_equal(_bits(s_dev), _bits(s_host))
        assert 0 < ctx.last_h2d_bytes < full // 4, (ctx.last_h2d_bytes, full)
        a_dev = ctx.analyze_frames(dclip, de, top, bot, 3, 17).cpu().numpy()
        a_host = ctx.analyze_frames(hclip, de, top, bot, 3, 17)
        assert np.array_equal(_bits(a_dev), _bits(a_host))
        fades = np.arange(0, 20, dtype=np.float32) * np.float32(0.1)
        e_dev = ctx.eval_fades(dclip, de, fades).cpu().numpy()
        e_host = ctx.eval_fades(hclip, de, fades)
        assert np.array_equal(_bits(e_dev), _bits(e_host))
        # in-place erase on host frames == in-place erase in HBM (8- and 16-bit)
        fd = np.stack([np.linspace(0, 1, n), np.linspace(1, 0, n)], axis=1).astype(np.float32)
        fd[5] = (0.5, 0.5)
        work_d = fr.clone()
        ctx.erase_logo(ab.yv12_clip(work_d, w, h, n, True, bits), raw, fd)
        work_h = host.copy()
        ctx.erase_logo(ab.yv12_clip(work_h, w, h, n, False, bits), raw, fd)
        assert np.array_equal(work_d.cpu().numpy(), work_h) and not np.array_equal(work_h, host)
        if bits == 8:
            sx, sy = imgx & ~1, imgy & ~1
            sw, sh = min(lw, w - sx) & ~1, min(lh, h - sy) & ~1
            a1, a2 = ctx.logo_scan(sw, sh, 12), ctx.logo_scan(sw, sh, 12)
            v1 = a1.add_frames(dclip, sx, sy)
            v2 = a2.add_frames(hclip, sx, sy)
            assert np.array_equal(v1, v2) and np.array_equal(a1.sums(), a2.sums())


def test_one_context_from_two_threads(ctx, oracle):
    """MT_NICE_FILTER: AviSynth may call GetFrame of one filter from several Prefetch threads.  Two host threads hammer ONE
    context with 1- and 2-frame calls (ctypes releases the GIL); every result equals the serial run."""
    import threading
    w, h, n = 256, 128, 24
    lg = synth.make_logo(64, 64)
    fr = synth.make_frames(40, n, w, h, device="cuda", logo=lg, imgx=160, imgy=32, logo_period=12)
    logo = ab.Logo.create(lg["data"], 64, 64, w, h, 160, 32).deint().create_mask(0.35)
    host = fr.cpu().numpy()
    hclip = ab.yv12_clip(host, w, h, n, False)
    dclip = ab.yv12_clip(fr, w, h, n, True)
    prm = ab.default_comb_params()
    ref_s = ctx.scan_frames(dclip, [logo]).cpu().numpy()
    ref_c = ctx.comb_frames(dclip, prm).cpu().numpy()
    errors = []

    def worker(tid):
        try:
            for rep in range(6):
                for i in range(tid, n, 2):
                    s = ctx.scan_frames(hclip, [logo], i, 1)
                    if not np.array_equal(_bits(s[0]), _bits(ref_s[i])):
                        errors.append(("scan", tid, i))
                    c = ctx.comb_frames(hclip, prm, i, 1)
                    if not np.array_equal(c[0], ref_c[i]):
                        errors.append(("comb", tid, i))
        except Exception as e:          # noqa
            errors.append(("exc", tid, repr(e)))

    ts = [threading.Thread(target=worker, args=(t,)) for t in range(2)]
    [t.start() for t in ts]
    [t.join() for t in ts]
    assert not errors, errors[:5]


@pytest.mark.parametrize("mode", ["1", "2"])
def test_fused_step_with_coresident_logo_kernel(oracle, monkeypatch, mode):
    """AMTK_SCAN_LITE=1: the logo evaluation of the fused step runs on a side stream UNDER the comb kernel (small-footprint
    kernel, taps from L2); =2: the same kernel on its own.  Not the default (DESIGN.md section 6) but kept tested: identical
    bits, 8- and 10-bit, device and host clips."""
    po = oracle
    w, h, n, imgx, imgy = 640, 360, 50, 500, 40
    lg = synth.make_logo(64, 64)
    monkeypatch.setenv("AMTK_SCAN_LITE", mode)
    c = ab.Context(0, torch.cuda.current_stream().cuda_stream)
    monkeypatch.delenv("AMTK_SCAN_LITE")
    try:
        f8 = _gen(7, n, w, h, logo=lg, imgx=imgx, imgy=imgy, logo_period=20)
        logo = ab.Logo.create(lg["data"], 64, 64, w, h, imgx, imgy).deint().create_mask(0.35)
        o = po.OracleLogo.create(lg["data"], 64, 64, w, h, imgx, imgy).deint().create_mask(0.35)
        prm = ab.default_comb_params()
        for rep in range(2):
            s, cn = c.scan_comb_frames(ab.yv12_clip(f8, w, h, n, True), [logo], prm)
        Y, U, V = synth.split_planes(f8, w, h)
        rs = np.stack([o.scan_frame(Y[i]) for i in range(n)])
        rc = po.or_comb_clip(Y, U, V, prm.as_list())
        assert np.array_equal(_bits(s.cpu().numpy()[:, 0]), _bits(rs)) and np.array_equal(cn.cpu().numpy(), rc)
        h8 = f8.cpu().numpy()                               # the descriptor holds a raw pointer: keep the array alive
        s2, c2 = c.scan_comb_frames(ab.yv12_clip(h8, w, h, n, False), [logo], prm)
        assert np.array_equal(_bits(s2[:, 0]), _bits(rs)) and np.array_equal(c2, rc)
        f16 = (f8.to(torch.int32) * 4 + (f8.to(torch.int32) & 3)).to(torch.int16).contiguous()
        p10 = ab.default_comb_params()
        p10.th_move_y, p10.th_shima_y, p10.th_lshima_y = 80, 48, 144
        s10, c10 = c.scan_comb_frames(ab.yv12_clip(f16, w, h, n, True, bits=10), [logo], p10)
        a16 = f16.cpu().numpy().view(np.uint16)
        Y10 = a16[:, :w * h].reshape(n, h, w)
        rs10 = np.stack([o.scan_frame(Y10[i], maxv=1023.0) for i in range(n)])
        assert np.array_equal(_bits(s10.cpu().numpy()[:, 0]), _bits(rs10))
    finally:
        c.close()


@pytest.mark.timeout(900)
@pytest.mark.parametrize("variant", ["ws", "cta_ring", "mma1", "mma2"])
def test_every_comb_kernel_variant_is_bit_exact(oracle, monkeypatch, variant):
    """The streaming pass exists in four forms: the default warp-stream kernel (comb_stream.cuh), the round-1 CTA-ring kernel
    (comb_kernels.cuh, AMTK_COMB_WS=0) and the two tensor-core forms (comb_mma.cuh: stencil as tcgen05.mma.kind::i8 with the
    TMA-staged tile as the MN-major operand; AMTK_COMB_MMA=1: one tile per CTA step, =2: two; every device-side wait of
    that kernel has a watchdog, so a protocol error fails the call instead of hanging the GPU).  All must return the spec
    oracle's counters bit for bit: ragged shapes (partial tile columns and rows, planes smaller than a tile, odd tile
    counts -> filler stream), extreme thresholds, edge rows, frame-range calls with a halo frame, and configs[1]/[2]
    geometry."""
    po = oracle
    env = {"ws": {}, "cta_ring": {"AMTK_COMB_WS": "0"}, "mma1": {"AMTK_COMB_MMA": "1"}, "mma2": {"AMTK_COMB_MMA": "2"}}[variant]
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    c = ab.Context(0, torch.cuda.current_stream().cuda_stream)
    for k in env:
        monkeypatch.delenv(k)
    try:
        prm = ab.default_comb_params()
        prm.th_move_y, prm.th_shima_y, prm.th_lshima_y = 1, 1, 2047
        prm.th_move_c, prm.th_shima_c, prm.th_lshima_c = 128, 700, 701
        for (w, h, n) in ((160, 34, 3), (128, 272, 5), (1952, 36, 2), (32, 1100, 2), (640, 360, 9)):
            fr = synth.make_frames(3, n, w, h, device="cuda", mode="interlaced")
            out = c.comb_frames(ab.yv12_clip(fr, w, h, n, True), prm).cpu().numpy()
            Y, U, V = synth.split_planes(fr, w, h)
            assert np.array_equal(out, po.or_comb_clip(Y, U, V, prm.as_list())), (variant, w, h)
        # maximum response everywhere: alternating 0 / 255 rows
        w, h = 256, 128
        fr = torch.zeros((2, w * h * 3 // 2), dtype=torch.uint8, device="cuda")
        fr[:, : w * h].view(2, h, w)[:, 0::2, :] = 255
        p2 = ab.default_comb_params()
        p2.th_shima_y, p2.th_lshima_y = 1530, 1531
        out = c.comb_frames(ab.yv12_clip(fr, w, h, 2, True), p2).cpu().numpy()
        assert out[0, 1] + out[0, 4] == (h - 4) * w and out[0, 2] + out[0, 5] == 0 and out[:, 0].sum() == 0
        # YUV420P10 (16-bit containers, 10 significant bits): "ws" = the warp-stream kernel's integer-lane form (default for
        # <= 10 bits), "cta_ring" = the round-1 fp32 kernel; ragged shapes incl. the merged U|V remainder tile and tiny planes
        p10 = ab.default_comb_params()
        p10.th_move_y, p10.th_shima_y, p10.th_lshima_y = 80, 48, 3000
        p10.th_move_c, p10.th_shima_c, p10.th_lshima_c = 200, 1, 6138
        for (w, h, n) in ((224, 136, 7), (320, 150, 5), (96, 62, 3), (1920, 64, 2), (64, 1100, 2)):
            f8 = synth.make_frames(2, n, w, h, device="cuda", mode="telecine")
            f16 = (f8.to(torch.int32) * 4 + (f8.to(torch.int32) & 3)).to(torch.int16).contiguous()
            f16[:, ::7] = 1023                                   # the largest legal sample, scattered
            clip10 = ab.yv12_clip(f16, w, h, n, True, bits=10)
            got = c.comb_frames(clip10, p10).cpu().numpy()
            a16 = f16.cpu().numpy().view(np.uint16)
            ysz, csz = w * h, (w // 2) * (h // 2)
            ref = po.or_comb_clip(a16[:, :ysz].reshape(n, h, w), a16[:, ysz:ysz + csz].reshape(n, h // 2, w // 2),
                                  a16[:, ysz + csz:].reshape(n, h // 2, w // 2), p10.as_list())
            assert np.array_equal(got, ref), (variant, "p10", w, h, np.argwhere(got != ref)[:5])
            if n > 4:
                part = np.concatenate([c.comb_frames(clip10, p10, 0, 3).cpu().numpy(), c.comb_frames(clip10, p10, 3, n - 3).cpu().numpy()])
                assert np.array_equal(part, ref), (variant, "p10 ranges", w, h)
        # BASELINE geometries with default thresholds, whole call and two range calls (halo frame)
        prm = ab.default_comb_params()
        for (w, h, n) in ((1920, 1080, 40), (1440, 1080, 18)):
            f8 = _gen(3, n, w, h, mode="telecine")
            clip = ab.yv12_clip(f8, w, h, n, True)
            got = c.comb_frames(clip, prm).cpu().numpy()
            Y, U, V = synth.split_planes(f8, w, h)
            ref = np.stack([po.or_comb_frame((Y[i], U[i], V[i]), (Y[max(i - 1, 0)], U[max(i - 1, 0)], V[max(i - 1, 0)]), prm.as_list(), "avx2")
                            for i in range(n)])
            assert np.array_equal(got, ref), (variant, w, h, np.argwhere(got != ref)[:5])
            part = np.concatenate([c.comb_frames(clip, prm, 0, 7).cpu().numpy(), c.comb_frames(clip, prm, 7, n - 7).cpu().numpy()])
            assert np.array_equal(part, ref), (variant, w, h, "ranges")
            assert ref[:, [1, 4]].sum() > 0 and ref[1:, 0].sum() > 0
    finally:
        c.close()
