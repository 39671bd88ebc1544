"""Encoder on the GPU (SURVEY.md 8a row a16).
 * Decision parity: at the same quantiser, on the same raw frames, the device encoder takes the decisions of
   the UNMODIFIED reference encoder (oracle/_ref/ref_encode, REALTIME_QUALITY as Salsify runs it): the records
   parsed back from both streams -- macroblock modes, sub-block modes, motion vectors, every quantised
   coefficient -- the loop-filter level and the reconstruction are equal, frame after frame.
 * RD parity at a target size (SURVEY 8d config 3): >= 30 raw 1080p frames, targets 20 000 / 60 000 bytes:
   bytes within 5 %, luma SSIM >= reference - 0.005, same frames, same aggregation.
 * Closed loop = the property the reference checks with export_decoder (encoder.hh:378): whoever decodes
   the emitted frames (CPU oracle, the unmodified reference decoder, this library's decoder) reconstructs
   exactly the raster the encoder kept as its LAST reference.
 * Encoder value semantics (copy, from a Decoder, export_decoder)."""
import os
import subprocess
import tempfile

import numpy as np
import pytest

import oracle_lib as O
import reference_outputs as R

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def synth(w, h, t, seed=7):
    """moving smooth pattern + a translating textured square + light noise"""
    rng = np.random.default_rng(seed)
    tex = rng.integers(0, 256, (64, 64)).astype(np.float32)
    tex = (tex + np.roll(tex, 1, 0) + np.roll(tex, 1, 1) + np.roll(tex, (1, 1), (0, 1))) / 4
    yy, xx = np.mgrid[0:h, 0:w].astype(np.float32)
    y = 128 + 60 * np.sin(0.03 * (xx + 3 * t)) * np.cos(0.02 * (yy + 2 * t))
    ox, oy = 20 + 3 * t, 30 + 2 * t
    y[oy:oy + 64, ox:ox + 64] = tex[:max(0, min(64, h - oy)), :max(0, min(64, w - ox))]
    y += np.random.default_rng(seed + t).integers(-2, 3, (h, w))
    cy, cx = np.mgrid[0:(h + 1) // 2, 0:(w + 1) // 2].astype(np.float32)
    u = 128 + 30 * np.sin(0.02 * (cx + t))
    v = 128 + 30 * np.cos(0.025 * (cy - t))
    return tuple(np.clip(a, 0, 255).astype(np.uint8) for a in (y, u, v))


def reference_encode(frames, w, h, qi=None, target=None, two_pass=False):
    """the unmodified reference encoder on raw frames: list of compressed frames.  Where oracle/_ref/ref_encode is not
    built, this library's encoder codes them and every frame must have the digest stored for the reference's."""
    k = R.key("ref_encode", w, h, qi, target, two_pass, frames)
    tool = R.tool("ref_encode")
    if tool is None:
        return _product_encode_as_reference(k, frames, w, h, qi, target, two_pass)
    with tempfile.TemporaryDirectory() as d:
        raw, out = os.path.join(d, "src.yuv"), os.path.join(d, "o.ivf")
        with open(raw, "wb") as f:
            for planes in frames:
                for p in planes:
                    f.write(np.ascontiguousarray(p).tobytes())
        env = dict(os.environ, REF_RAW=raw)
        if target is not None:
            env["REF_TARGET"] = str(target)
        if two_pass:
            env["REF_TWO_PASS"] = "1"
        r = subprocess.run([tool, out, str(w), str(h), str(len(frames)), "100000", str(qi or 0)], env=env,
                           capture_output=True, text=True)
        assert r.returncode == 0, r.stderr[-400:]
        _, _, chunks = O.read_ivf(open(out, "rb").read())
    return R.check(k, chunks)


def _product_encode_as_reference(k, frames, w, h, qi, target, two_pass):
    from alfalfa_b200 import Context, Encoder
    want = R.stored(k)
    ctx = Context(w, h, max_frames=32)
    enc = Encoder(ctx)
    if two_pass:
        enc.set_two_pass(True)
    chunks = []
    for t, planes in enumerate(frames):
        blob = enc.encode_with_target_size(*planes, target)[0] if target is not None else enc.encode_with_quantizer(*planes, qi)
        assert R.digest(blob) == want[t], "frame %d: %d bytes vs %d bytes of the reference encoder (digest differs)" % (
            t, len(blob), want[t][0])
        chunks.append(blob)
    assert len(chunks) == len(want)
    del enc
    ctx.close()
    return chunks


def dense_coefficients(mbs, tok):
    """[n_mbs, 25, 16] quantised coefficients from a record / token pair (the pool order is not compared)"""
    out = np.zeros((len(mbs), 25, 16), np.int32)
    for i, m in enumerate(mbs):
        t = tok[m["tok_off"]:m["tok_off"] + m["tok_cnt"]]
        out[i, (t >> 20) & 31, (t >> 16) & 15] = (t & 0xFFFF).astype(np.int16)
    return out


def assert_same_decisions(pa, pb, what):
    """records of the same frame parsed from two streams: same decisions?"""
    da, db = pa.desc, pb.desc
    assert (da.key_frame, da.loop_filter_level, list(da.quant)) == (db.key_frame, db.loop_filter_level, list(db.quant)), what
    (ma, ta, _), (mb, tb, _) = pa.arrays(), pb.arrays()
    assert np.array_equal(ma["ref_frame"], mb["ref_frame"]), "%s: intra / inter decisions differ at %s" % (
        what, np.nonzero(ma["ref_frame"] != mb["ref_frame"])[0][:8])
    intra = ma["ref_frame"] == 0
    for field in ("y_mode", "uv_mode", "b_modes"):
        bad = np.nonzero(intra & (ma[field] != mb[field]))[0]
        assert bad.size == 0, "%s: %s differs at macroblocks %s: %s vs %s" % (what, field, bad[:8], ma[field][bad[:8]], mb[field][bad[:8]])
    for field in ("mv_x", "mv_y"):
        bad = np.nonzero(~intra & (ma[field] != mb[field]))[0]
        assert bad.size == 0, "%s: %s differs at macroblocks %s: %s vs %s" % (what, field, bad[:8], ma[field][bad[:8]], mb[field][bad[:8]])
    ca, cb = dense_coefficients(ma, ta), dense_coefficients(mb, tb)
    bad = np.nonzero((ca != cb).any(axis=(1, 2)))[0]
    assert bad.size == 0, "%s: coefficients differ at macroblocks %s" % (what, bad[:8])


@pytest.mark.parametrize("size,n,qi", [((320, 240), 8, 40), ((176, 144), 6, 12), ((640, 368), 6, 70), ((1920, 1080), 3, 90)])
def test_decisions_equal_the_reference_encoder(size, n, qi):
    from alfalfa_b200 import Context, Decoder, Encoder
    w, h = size
    frames = [synth(w, h, t) for t in range(n)]
    ref = reference_encode(frames, w, h, qi=qi)
    ctx = Context(w, h, max_frames=32)
    enc = Encoder(ctx)
    da, db, dd = Decoder(ctx), Decoder(ctx), Decoder(ctx)  # dd follows (decodes) the REFERENCE stream
    for t in range(n):
        blob = enc.encode_with_quantizer(*frames[t], qi)
        assert_same_decisions(da.parse_frame(blob), db.parse_frame(ref[t]), "frame %d of %dx%d q%d" % (t, w, h, qi))
        # the reference's stream decodes to the raster this encoder kept
        rec = enc.reconstruction()
        _, theirs = dd.get_frame_output(ref[t])
        assert all(np.array_equal(a, b) for a, b in zip(theirs.planes(), rec.planes())), "frame %d: reconstruction differs" % t
        theirs.release()
        rec.release()
        # same records and the reference's own header rules (serializer.h RefWriterState): the same bytes
        assert blob == ref[t], "frame %d: %d bytes vs %d bytes of the reference, first difference at byte %d" % (
            t, len(blob), len(ref[t]), next((i for i, (a, b) in enumerate(zip(blob, ref[t])) if a != b), -1))
    del enc, da, db, dd
    ctx.close()


def test_rd_parity_at_target_size_1080p():
    """SURVEY 8d config 3: encode_with_target_size at 20 000 and 60 000 bytes per frame over 30 raw 1080p
    frames next to the reference encoder: bytes within 5 %, SSIM >= reference - 0.005 (xc-enc-ssim.test:23),
    both measured the same way: every stream decoded by this library's decoder, device SSIM of the shown
    luma against the source, mean over the same 30 frames."""
    from alfalfa_b200 import Context, Decoder, Encoder
    import bench
    w, h, n = 1920, 1080, 30
    frames = [bench.synth_1080p(t) for t in range(n)]
    ctx = Context(w, h, max_frames=32)
    src = ctx.alloc_frame()

    def mean_ssim(chunks):
        dec = Decoder(ctx)
        vals = []
        for t, c in enumerate(chunks):
            _, r = dec.get_frame_output(c)
            src.upload(*frames[t])
            vals.append(r.ssim(src))
            r.release()
        return float(np.mean(vals))

    for target in (20000, 60000):
        ref = reference_encode(frames, w, h, target=target)
        enc = Encoder(ctx)
        ours, qis = [], []
        for t in range(n):
            blob, qi = enc.encode_with_target_size(*frames[t], target)
            ours.append(blob)
            qis.append(qi)
        del enc
        ref_bytes, our_bytes = sum(map(len, ref)), sum(map(len, ours))
        ref_ssim, our_ssim = mean_ssim(ref), mean_ssim(ours)
        print("target %d: bytes ours %d reference %d (%.2f %%), SSIM ours %.5f reference %.5f, qi %s" % (
            target, our_bytes, ref_bytes, 100.0 * (our_bytes - ref_bytes) / ref_bytes, our_ssim, ref_ssim, qis))
        assert abs(our_bytes - ref_bytes) <= 0.05 * ref_bytes, (target, our_bytes, ref_bytes)
        assert our_ssim >= ref_ssim - 0.005, (target, our_ssim, ref_ssim)
        # in fact the same quantiser search on the same estimates picks the same indices and emits the same bytes
        pd = Decoder(ctx)
        ref_qis = [pd.parse_frame(c).desc.quant[1] for c in ref]  # y_ac of segment 0
        pd = Decoder(ctx)
        our_qis = [pd.parse_frame(c).desc.quant[1] for c in ours]
        assert our_qis == ref_qis, (our_qis, ref_qis)
        da, db = Decoder(ctx), Decoder(ctx)
        for t in range(n):
            pa, pb = da.parse_frame(ours[t]), db.parse_frame(ref[t])
            if ours[t] != ref[t]:
                assert_same_decisions(pa, pb, "target %d frame %d" % (target, t))
                assert False, "target %d frame %d: same decisions, different bytes (%d vs %d, first difference at %d)" % (
                    target, t, len(ours[t]), len(ref[t]), next((i for i, (a, b) in enumerate(zip(ours[t], ref[t])) if a != b), -1))
        # the compact writer (same decisions, only the header updates that pay, 8 partitions) is never larger
        enc = Encoder(ctx)
        enc.set_writer(1)
        compact = [enc.encode_with_target_size(*frames[t], target)[0] for t in range(n)]
        del enc
        print("           compact writer: %d bytes, SSIM %.5f" % (sum(map(len, compact)), mean_ssim(compact)))
    src.release()
    ctx.close()


def test_first_inter_frame_estimates_price_vectors_at_zero():
    """The reference fills its motion-vector cost tables at the start of the first FULL inter-frame pass
    (encode_inter.cc:601-602), so the size estimates of the first inter frame price every vector at 0 and the
    sampled motion search runs off to long vectors; target 45 000 on the bench clip is where that decides the
    quantiser (qi 102; 100 with priced vectors).  Every frame must equal the reference encoder's."""
    from alfalfa_b200 import Context, Encoder
    import bench
    w, h, n, target = 1920, 1080, 6, 45000
    frames = [bench.synth_1080p(t) for t in range(n)]
    ref = reference_encode(frames, w, h, target=target)
    ctx = Context(w, h, max_frames=32)
    enc = Encoder(ctx)
    for t in range(n):
        blob, qi = enc.encode_with_target_size(*frames[t], target)
        assert blob == ref[t], "frame %d (qi %d): %d bytes vs %d of the reference" % (t, qi, len(blob), len(ref[t]))
    del enc
    ctx.close()


def test_encoder_value_semantics():
    """Encoder( const Encoder & ), Encoder( const Decoder &, ... ), export_decoder (encoder.hh:346-382): a copy
    encodes the same next frame as the original, concurrently (salsify-sender.cc:492-518); export_decoder is a
    Decoder equal to one that decoded the emitted frames; an Encoder made from that Decoder continues the stream."""
    import threading
    from alfalfa_b200 import Context, Decoder, Encoder
    w, h = 320, 240
    ctx = Context(w, h, max_frames=48)
    enc = Encoder(ctx)
    dec = Decoder(ctx)
    for t in range(3):
        blob = enc.encode_with_quantizer(*synth(w, h, t), 50)
        _, r = dec.get_frame_output(blob)
        r.release()
    exported = enc.export_decoder()
    assert exported == dec and exported.get_hash() == dec.get_hash()
    assert enc.minihash() == dec.minihash()
    a, b = enc.copy(), enc.copy()
    nxt = synth(w, h, 3)
    out = {}

    def run(name, e, qi):
        out[name] = e.encode_with_quantizer(*nxt, qi)
    th = [threading.Thread(target=run, args=("a", a, 60)), threading.Thread(target=run, args=("b", b, 20))]
    [x.start() for x in th]
    [x.join() for x in th]
    assert out["a"] == enc.copy().encode_with_quantizer(*nxt, 60)
    assert out["b"] == enc.copy().encode_with_quantizer(*nxt, 20) and len(out["b"]) > len(out["a"])
    # the original is untouched by what its copies did
    assert enc.export_decoder() == dec
    cont = Encoder.from_decoder(ctx, dec)
    blob = cont.encode_with_quantizer(*nxt, 60)
    assert (blob[0] & 1) == 1  # continues with an inter frame
    # not byte-equal to out["a"] in general: an Encoder built from a Decoder has no previous loop-filter level
    # (encoder.hh:144, Optional) and searches from level 0 (encoder.cc:475-487), a copy searches around the last one;
    # what must hold is the closed loop below
    _, r = dec.get_frame_output(blob)
    assert cont.export_decoder() == dec
    r.release()
    del enc, a, b, cont, dec, exported
    ctx.close()


def reference_decode_shown(ivf):
    """digest of what the unmodified reference decoder shows for an IVF stream (ref_dump shown)"""
    def run():
        with tempfile.NamedTemporaryFile(suffix=".ivf") as f:
            f.write(ivf)
            f.flush()
            r = subprocess.run([R.tool("ref_dump"), "shown", f.name], capture_output=True)
        assert r.returncode == 0, r.stderr[-400:]
        return [r.stdout]
    return R.expected(R.key("ref_dump shown", ivf), run if R.tool("ref_dump") else None)[0]


def psnr(a, b):
    mse = np.mean((a.astype(np.float64) - b.astype(np.float64)) ** 2)
    return 99.0 if mse == 0 else 10 * np.log10(255.0 ** 2 / mse)


@pytest.mark.parametrize("size", [(320, 240), (176, 144), (200, 120)])
def test_closed_loop_against_oracle_reference_and_own_decoder(size):
    from alfalfa_b200 import Context, Decoder, Encoder, write_ivf
    w, h = size
    ctx = Context(w, h, max_frames=32)
    enc = Encoder(ctx)
    dec = Decoder(ctx)
    od = O.OracleDecoder(w, h)
    frames, recon_display = [], []
    for t in range(6):
        y, u, v = synth(w, h, t)
        blob = enc.encode_with_quantizer(y, u, v, 40 if t else 30)
        frames.append(blob)
        assert (blob[0] & 1) == (0 if t == 0 else 1)  # first frame key, then inter frames
        rec = enc.reconstruction()
        rp = rec.planes()
        want = od.decode(blob)
        assert want["shown"]
        for g, w_ in zip(rp, want["planes"]):
            assert np.array_equal(g, w_), "frame %d: oracle decode differs from the encoder's reconstruction" % t
        shown, mine = dec.get_frame_output(blob)
        assert all(np.array_equal(a, b) for a, b in zip(mine.planes(), rp))
        assert psnr(rp[0][:h, :w], y) > 30.0, "frame %d PSNR %.1f" % (t, psnr(rp[0][:h, :w], y))
        recon_display.append(rec.display_bytes())
        rec.release()
        mine.release()
    # motion-compensated frames (coarser quantiser, mostly noise left to code) stay below the key frame
    assert sum(len(f) for f in frames[1:]) / 5 < len(frames[0])
    # the unmodified reference decoder agrees as well
    assert R.digest(b"".join(recon_display)) == reference_decode_shown(write_ivf(w, h, frames))
    del enc, dec
    ctx.close()


def test_target_size_search_and_rate_monotonicity():
    from alfalfa_b200 import Context, Encoder
    w, h = 320, 240
    ctx = Context(w, h, max_frames=32)
    sizes = {}
    for qi in (10, 40, 90):
        enc = Encoder(ctx)
        sizes[qi] = len(enc.encode_with_quantizer(*synth(w, h, 0), qi))
        del enc
    assert sizes[10] > sizes[40] > sizes[90]
    enc = Encoder(ctx)
    target = (sizes[40] + sizes[90]) // 2
    blob, qi = enc.encode_with_target_size(*synth(w, h, 0), target)
    # the search runs on the sampled estimate (size_estimation.cc): the index is the smallest whose ESTIMATE fits
    probe = Encoder(ctx)
    assert probe.estimate_frame_size(*synth(w, h, 0), qi) <= target < probe.estimate_frame_size(*synth(w, h, 0), qi - 1)
    assert 10 < qi <= 127 and len(blob) < 2 * target
    blob2, qi2 = enc.encode_with_target_size(*synth(w, h, 1), target // 3)
    assert (blob2[0] & 1) == 1 and abs(qi2 - qi) <= 16  # inter frame, search window last_qi +- 16
    del enc, probe
    ctx.close()


@pytest.mark.parametrize("w,h,n,target", [(320, 240, 5, 2500), (176, 144, 4, 1200), (640, 368, 3, 8000)])
def test_searches_in_one_launch_equal_candidate_by_candidate(w, h, n, target):
    """The target-size search codes every probe it can still reach in one k_enc_rd launch (33 sampled passes, or the
    next three levels of the bisection tree for the first frame's wider range), the loop-filter search its trials in
    one k_loopfilter launch.  Same session with VP8GPU_ENC_SPECULATE=0 (one launch per candidate, the round-1 order):
    same bytes, same quantisers, same loop-filter levels, same SSIM, same Decoder state -- and fewer launches."""
    import json
    import sys
    worker = os.path.join(ROOT, "tests", "encoder_search_worker.py")
    res = {}
    for mode in ("1", "0"):
        r = subprocess.run([sys.executable, worker, str(w), str(h), str(n), str(target)], env=dict(os.environ, VP8GPU_ENC_SPECULATE=mode),
                           capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, (r.stdout + r.stderr)[-1500:]
        res[mode] = json.loads(r.stdout.strip().splitlines()[-1])
    assert res["1"]["frames"] == res["0"]["frames"]
    for mode in ("1", "0"):  # vp8gpu_encoder_timeline: every phase a time, the parts that run one after the other within the whole
        tl = res[mode]["timeline"]
        assert all(v >= 0 for v in tl.values()) and tl["total"] > 0 and tl["full_pass"] > 0
        assert tl["upload"] + tl["estimates_launch"] + tl["estimates_walk"] + tl["full_pass"] + tl["loop_filter_search"] + tl["state_update"] <= tl["total"] * 1.001 + 0.05
    assert res["1"]["launches"] < res["0"]["launches"], (res["1"]["launches"], res["0"]["launches"])


def ssim_x264(a, b):
    """util/ssim.cc -> x264 pixel_ssim_wxh / window count, restated with numpy: integer sums over every
    8x8 window at a 4-pixel step (oracle/ref_shim/ssim_stub.cc), float32 ratio, mean in float64"""
    a, b = a.astype(np.int64), b.astype(np.int64)
    H, W = a.shape

    def blocks(x):  # sums over 4x4 blocks
        return x.reshape(H // 4, 4, W // 4, 4).sum(axis=(1, 3))

    def win(x):  # 2x2 blocks = one 8x8 window
        return x[:-1, :-1] + x[:-1, 1:] + x[1:, :-1] + x[1:, 1:]
    s1, s2 = win(blocks(a)), win(blocks(b))
    ss, s12 = win(blocks(a * a + b * b)), win(blocks(a * b))
    c1 = int(.01 * .01 * 255 * 255 * 64 + .5)
    c2 = int(.03 * .03 * 255 * 255 * 64 * 63 + .5)
    vars_, covar = ss * 64 - s1 * s1 - s2 * s2, s12 * 64 - s1 * s2
    num = (2 * s1 * s2 + c1).astype(np.float32) * (2 * covar + c2).astype(np.float32)
    den = (s1 * s1 + s2 * s2 + c1).astype(np.float32) * (vars_ + c2).astype(np.float32)
    return float((num / den).astype(np.float64).mean())


def test_device_ssim_matches_the_restated_x264_ssim():
    from alfalfa_b200 import Context
    w, h = 320, 240
    ctx = Context(w, h, max_frames=8)
    rng = np.random.default_rng(3)
    for trial in range(4):
        y0, u0, v0 = synth(w, h, trial)
        noise = rng.integers(-(4 << trial), (4 << trial) + 1, y0.shape)
        y1 = np.clip(y0.astype(np.int64) + noise, 0, 255).astype(np.uint8)
        a, b = ctx.alloc_frame(), ctx.alloc_frame()
        a.upload(y0, u0, v0)
        b.upload(y1, u0, v0)
        got = a.ssim(b)
        want = ssim_x264(y0, y1)
        assert abs(got - want) < 2e-6, (trial, got, want)
        assert abs(a.ssim(a) - 1.0) < 1e-9
        a.release()
        b.release()
    ctx.close()


def test_loop_filter_choice_and_minimum_ssim():
    """Encoder::apply_best_loopfilter_settings / encode_with_minimum_ssim: the reported SSIM is the SSIM of
    the kept reconstruction against the (edge-extended) source, the frame header carries the chosen level,
    and the minimum-SSIM search returns the coarsest quantiser that still reaches the bound."""
    from alfalfa_b200 import Context, Decoder, Encoder
    w, h = 320, 240
    ctx = Context(w, h, max_frames=32)
    enc = Encoder(ctx)
    od = O.OracleDecoder(w, h)
    src = ctx.alloc_frame()
    for t in range(4):
        y, u, v = synth(w, h, t)
        blob = enc.encode_with_quantizer(y, u, v, 60)
        st = enc.stats()
        rec = enc.reconstruction()
        src.upload(y, u, v)
        assert abs(st["ssim"] - rec.ssim(src)) < 1e-9
        want = od.decode(blob)
        assert od.parsed().desc.loop_filter_level == st["loop_filter_level"]
        for g, w_ in zip(rec.planes(), want["planes"]):
            assert np.array_equal(g, w_)
        rec.release()
    # estimate_frame_size: 16 x the size of the 1/16 sample, and leaves the encoder untouched
    y, u, v = synth(w, h, 4)
    before = enc.stats()
    hash_before = enc.minihash()
    est = enc.estimate_frame_size(y, u, v, 50)
    assert enc.stats() == before and enc.minihash() == hash_before
    twin_blob = enc.encode_with_quantizer(y, u, v, 50)
    assert est % 16 == 0 and 0.3 * len(twin_blob) < est < 3 * len(twin_blob)
    od.decode(twin_blob)
    # minimum SSIM: reached, and one step coarser would not reach it (checked with a twin encoder state)
    y, u, v = synth(w, h, 5)
    target = 0.93
    blob, qi = enc.encode_with_minimum_ssim(y, u, v, target)
    st = enc.stats()
    assert st["y_ac_qi"] == qi and (st["ssim"] >= target or qi == 0)
    want = od.decode(blob)
    rec = enc.reconstruction()
    for g, w_ in zip(rec.planes(), want["planes"]):
        assert np.array_equal(g, w_)
    rec.release()
    src.release()
    del enc
    ctx.close()


@pytest.mark.parametrize("name", ["04b68b0a642d8285303d2b8884fc374e09d28ae9", "07b5eb1e9741d90027c46166eaaff566c6bf934f",
                                  "a4dace04a77fc9f969a8d7a645c99c0271f1f73e", "ced8ea7239e3c4ee32ed7ed6c9ff9cdfbaba3ae4",
                                  "e3bc5f0c53d5efd6f2b1ea1a17ed1ee9bde5ea48"])
def test_encoder_built_from_a_decoder_in_any_state_stays_in_step(name):
    """Encoder( const Decoder & ) (encoder.hh:350-351) after a libvpx stream: the decoder's state carries updated mode /
    motion-vector probabilities, loop-filter adjustments, segmentation.  The frames the Encoder then emits must be
    coded against that state: a receiver that decodes them equals export_decoder() after every frame."""
    from alfalfa_b200 import Context, Decoder, Encoder
    from conftest import GOLDEN_DIR, golden_vectors
    full = [n for n in golden_vectors() if n.startswith(name[:8])][0]
    w, h, chunks = O.read_ivf(open(os.path.join(GOLDEN_DIR, full), "rb").read())
    ctx = Context(w, h, max_frames=24)
    rx = Decoder(ctx)
    for c in chunks[:10]:
        rx.get_frame_output(c)
    enc = Encoder.from_decoder(ctx, rx)
    for t in range(3):
        frame = enc.encode_with_quantizer(*synth(w, h, t), 36 + 8 * t)
        assert frame[0] & 1, "an Encoder built from a Decoder continues with inter frames"
        rx.get_frame_output(frame)
        assert rx == enc.export_decoder(), "frame %d" % t
    ctx.close()


def _noisy(w, h, t, amp):
    y, u, v = synth(w, h, t)
    rng = np.random.default_rng(100 + t)
    return tuple(np.clip(p.astype(np.int32) + rng.integers(-amp, amp + 1, p.shape), 0, 255).astype(np.uint8) for p in (y, u, v))


@pytest.mark.parametrize("w,h,qi,amp,n", [(64, 64, 40, 20, 2), (176, 144, 70, 40, 2), (175, 143, 60, 35, 3), (320, 240, 110, 60, 2),
                                        (640, 368, 40, 30, 2)])
def test_two_pass_key_frames_equal_the_reference_encoder(w, h, qi, amp, n):
    """Encoder( ..., two_pass = true, ... ): the key frame's second pass with trellis quantisation (k_enc_rd<true>:
    Encoder::trellis_quantize, check_reset_y2, encoder.cc:198-408; token contexts from requantised neighbours; the block
    types and Y2 flags the first pass left behind, encode_intra.cc:58-66, 181-184) -- frames byte-identical to the
    unmodified reference's (REF_TWO_PASS), noisy sources so that the trellis has something to decide"""
    from alfalfa_b200 import Context, Decoder, Encoder
    frames = [_noisy(w, h, t, amp) for t in range(n)]
    want = reference_encode(frames, w, h, qi=qi, two_pass=True)
    one_pass = reference_encode(frames[:1], w, h, qi=qi)
    ctx = Context(w, h, max_frames=16)
    enc = Encoder(ctx)
    enc.set_two_pass(True)
    got = [enc.encode_with_quantizer(*f, qi) for f in frames]
    assert got == want
    assert got[0] != one_pass[0], "the second pass changed nothing: the case does not exercise the trellis"
    rx = Decoder(ctx)
    for c in got:
        rx.get_frame_output(c)
    assert rx == enc.export_decoder()
    ctx.close()
