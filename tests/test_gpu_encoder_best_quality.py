"""Encoder at BEST_QUALITY (encoder.hh:56-60), ExCamera's xc-enc default, against the UNMODIFIED reference encoder built
with the same setting (oracle/_ref/ref_encode_best and ref_reencode_best, oracle/ref_best.mk).

At BEST every inter-frame macroblock runs the B_PRED trial (encode_intra.cc:98-102) and the NEWMV diamond search
(encode_inter.cc:278-285), and no frame remembers its quantiser or loop-filter level (encoder.cc:164-167): every
target-size search bisects over [4, 127], every loop-filter search walks up from level 0.  The B_PRED trial of a
macroblock prices its sub-block modes in the context of the modes its neighbours left in the frame object -- for an
inter neighbour those of its own losing trial.  Every case compares bytes (and, at fixed quantisers, every decision and
the reconstruction) with the reference's, frame after frame.  The reference's digests for these cases are kept in a store
of their own (tests/reference_outputs_best.py); the REALTIME inputs some cases start from come from reference_outputs.

This file also runs on the CPU under the SIMT emulator (tests/test_simt_best_quality.py), without the 1080p case."""
import os
import subprocess
import tempfile

import numpy as np
import pytest

import oracle_lib as O
import reference_outputs as R
import reference_outputs_best as B
from test_gpu_encoder import _noisy, assert_same_decisions, synth
from test_gpu_reencode import _decoded_targets, _full_name, _golden, ivf_bytes, make_case, reference_state_after

pytestmark = pytest.mark.gpu


def reference_encode_best(frames, w, h, qi=None, target=None, two_pass=False):
    """ref_encode_best: list of compressed frames.  Where the tool is not built, this library's encoder
    at BEST codes them and every frame must have the digest stored for the reference's."""
    k = R.key("ref_encode", w, h, qi, target, two_pass, frames, "best")
    tool = R.tool("ref_encode_best")
    if tool is None:
        return _product_encode(k, frames, w, h, qi, target, two_pass)
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
    return B.check(k, chunks)


def _product_encode(k, frames, w, h, qi, target, two_pass):
    from alfalfa_b200 import Context, Encoder
    want = B.stored(k)
    ctx = Context(w, h, max_frames=32)
    enc = Encoder(ctx, quality="best")
    enc.set_two_pass(two_pass)
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


def reference_reencode_best(w, h, targets, pred_chunks, state_blob, kf_q_weight, extra_frame_chunk):
    """ref_reencode_best: the reference's Encoder::reencode; digests of the emitted frames"""
    def run():
        with tempfile.TemporaryDirectory() as d:
            raw, pred, state, out = (os.path.join(d, n) for n in ("t.yuv", "p.ivf", "s.bin", "o.ivf"))
            with open(raw, "wb") as f:
                for planes in targets:
                    for p in planes:
                        f.write(np.ascontiguousarray(p).tobytes())
            open(pred, "wb").write(ivf_bytes(w, h, pred_chunks))
            open(state, "wb").write(state_blob)
            r = subprocess.run([R.tool("ref_reencode_best"), out, str(w), str(h), raw, pred, state, repr(kf_q_weight),
                                str(int(extra_frame_chunk))], capture_output=True, text=True)
            assert r.returncode == 0, r.stderr[-400:]
            return O.read_ivf(open(out, "rb").read())[2]
    k = R.key("ref_reencode", w, h, targets, pred_chunks, state_blob, kf_q_weight, bool(extra_frame_chunk), "best")
    return B.expected(k, run if R.tool("ref_reencode_best") else None)


def product_reencode_best(w, h, targets, pred_chunks, state_blob, kf_q_weight, extra_frame_chunk):
    """this library's Encoder::reencode at BEST from the same state: (emitted frames, receiver in step)"""
    from alfalfa_b200 import Context, Decoder, Encoder
    ctx = Context(w, h, max_frames=24)
    pred_decoder = Decoder(ctx)
    prediction_frames = []
    for c in pred_chunks:
        pf = pred_decoder.parse_frame(c, keep_labels=True)
        pred_decoder.decode_frame(pf)
        prediction_frames.append(pf)
    enc = Encoder.from_decoder(ctx, Decoder.deserialize(ctx, state_blob), quality="best")
    frames = enc.reencode(targets, prediction_frames, kf_q_weight, extra_frame_chunk)
    rx = Decoder.deserialize(ctx, state_blob)
    for c in frames:
        rx.get_frame_output(c)[1].release()
    in_step = rx == enc.export_decoder()
    del enc, rx, pred_decoder, prediction_frames
    ctx.close()
    return frames, in_step


def first_difference(a, b):
    return next((i for i, (x, y) in enumerate(zip(a, b)) if x != y), min(len(a), len(b)))


@pytest.mark.parametrize("w,h,n,qi", [(176, 144, 6, 12), (320, 240, 6, 40), (640, 368, 6, 70), (175, 143, 6, 56)])
def test_best_decisions_equal_the_reference_encoder(w, h, n, qi):
    """encode_with_quantizer at BEST: records, reconstruction and bytes of every frame equal the reference's"""
    from alfalfa_b200 import Context, Decoder, Encoder
    frames = [synth(w, h, t) for t in range(n)]
    ref = reference_encode_best(frames, w, h, qi=qi)
    ctx = Context(w, h, max_frames=32)
    enc = Encoder(ctx, quality="best")
    da, db, dd = Decoder(ctx), Decoder(ctx), Decoder(ctx)  # dd follows (decodes) the reference's stream
    inter_bpred = 0
    for t in range(n):
        blob = enc.encode_with_quantizer(*frames[t], qi)
        pa, pb = da.parse_frame(blob), db.parse_frame(ref[t])
        assert_same_decisions(pa, pb, "BEST frame %d of %dx%d q%d" % (t, w, h, qi))
        if t:
            m = pa.arrays()[0]
            inter_bpred += int(np.sum((m["ref_frame"] == 0) & (m["y_mode"] == 4)))  # VP8GPU_B_PRED
        rec = enc.reconstruction()
        _, theirs = dd.get_frame_output(ref[t])
        assert all(np.array_equal(a, b) for a, b in zip(theirs.planes(), rec.planes())), "frame %d: reconstruction differs" % t
        theirs.release()
        rec.release()
        assert blob == ref[t], "frame %d: %d bytes vs %d bytes of the reference, first difference at byte %d" % (
            t, len(blob), len(ref[t]), first_difference(blob, ref[t]))
    print("%dx%d q%d: %d B_PRED macroblocks in inter frames" % (w, h, qi, inter_bpred))
    del enc, da, db, dd
    ctx.close()


@pytest.mark.parametrize("target", [1500, 4000])
def test_best_target_size_searches_start_from_scratch(target):
    """encode_with_target_size at BEST over 6 frames: every frame bisects over [4, 127] and walks the loop-filter levels up
    from 0; the chosen quantisers, loop-filter levels and bytes equal the reference's"""
    from alfalfa_b200 import Context, Encoder
    w, h, n = 320, 240, 6
    frames = [synth(w, h, t) for t in range(n)]
    ref = reference_encode_best(frames, w, h, target=target)
    ctx = Context(w, h, max_frames=32)
    enc = Encoder(ctx, quality="best")
    od = O.OracleDecoder(w, h)
    for t in range(n):
        blob, qi = enc.encode_with_target_size(*frames[t], target)
        od.decode(blob)
        st = enc.stats()
        assert (st["y_ac_qi"], st["loop_filter_level"]) == (qi, od.parsed().desc.loop_filter_level)
        assert blob == ref[t], "frame %d (qi %d): %d bytes vs %d of the reference, first difference at byte %d" % (
            t, qi, len(blob), len(ref[t]), first_difference(blob, ref[t]))
    del enc
    ctx.close()


def test_best_two_pass_key_frame():
    """Encoder( w, h, two_pass = true, BEST_QUALITY ): the trellis pass of the key frame, then BEST inter frames"""
    from alfalfa_b200 import Context, Encoder
    w, h, qi = 176, 144, 70
    frames = [_noisy(w, h, t, 40) for t in range(3)]
    want = reference_encode_best(frames, w, h, qi=qi, two_pass=True)
    ctx = Context(w, h, max_frames=16)
    enc = Encoder(ctx, quality="best")
    enc.set_two_pass(True)
    got = [enc.encode_with_quantizer(*f, qi) for f in frames]
    for t, (a, b) in enumerate(zip(got, want)):
        assert a == b, "frame %d: %d vs %d bytes, first difference at byte %d" % (t, len(a), len(b), first_difference(a, b))
    del enc
    ctx.close()


def test_best_1080p_key_and_two_inter_frames():
    """the bench clip at 1080p: a key frame and two inter frames at BEST, byte for byte"""
    from alfalfa_b200 import Context, Encoder
    import bench
    w, h, qi = 1920, 1080, 60
    frames = [bench.synth_1080p(t) for t in range(3)]
    want = reference_encode_best(frames, w, h, qi=qi)
    ctx = Context(w, h, max_frames=32)
    enc = Encoder(ctx, quality="best")
    for t in range(3):
        blob = enc.encode_with_quantizer(*frames[t], qi)
        assert blob == want[t], "frame %d: %d vs %d bytes, first difference at byte %d" % (
            t, len(blob), len(want[t]), first_difference(blob, want[t]))
    del enc
    ctx.close()


@pytest.mark.parametrize("kf_q_weight", [1.0, 0.5])
@pytest.mark.parametrize("extra_frame_chunk", [False, True])
def test_best_reencode_equals_the_reference(extra_frame_chunk, kf_q_weight):
    """Encoder::reencode at BEST on the chunks tests/test_gpu_reencode.py builds: a whole chunk (options 1 + 4: the key
    frame through the BEST decision loop) and an extra-frame chunk (options 2 + 4)"""
    w, h, n = 176, 144, 4
    targets, pred, state = make_case(w, h, n, qi_a=40, qi_b=64 if not extra_frame_chunk else 56)
    want = reference_reencode_best(w, h, targets, pred, state, kf_q_weight, extra_frame_chunk)
    got, in_step = product_reencode_best(w, h, targets, pred, state, kf_q_weight, extra_frame_chunk)
    assert len(got) == len(want) == (n - 1 if extra_frame_chunk else n)
    for i, (a, b) in enumerate(zip(got, want)):
        assert R.digest(a) == b, "frame %d: %d vs %d bytes" % (i, len(a), b[0])
    assert in_step


def test_best_reencode_on_a_libvpx_prediction_stream():
    """a whole chunk whose prediction frames libvpx wrote (SPLITMV, intra macroblocks in inter frames, loop-filter
    deltas), re-encoded at BEST from the state another libvpx stream left"""
    pw, ph, prev_chunks = _golden(_full_name("04b68b0a"))
    w, h, chunks = _golden(_full_name("07b5eb1e"))
    assert (pw, ph) == (w, h)
    chunks = chunks[:10]
    state = reference_state_after(w, h, prev_chunks, len(prev_chunks))
    targets = _decoded_targets(w, h, chunks)
    want = reference_reencode_best(w, h, targets, chunks, state, 0.75, False)
    got, in_step = product_reencode_best(w, h, targets, chunks, state, 0.75, False)
    assert len(got) == len(want) == len(chunks)
    for i, (a, b) in enumerate(zip(got, want)):
        assert R.digest(a) == b, "frame %d: %d vs %d bytes" % (i, len(a), b[0])
    assert in_step


def test_best_closed_loop_copies_and_setting_rules():
    """what a caller relies on at BEST: every emitted frame decodes (CPU oracle) to the encoder's reconstruction and
    export_decoder() equals a decoder fed the frames; stats() reports the level and quantiser of the last frame; a copy
    inherits BEST; an Encoder built from a Decoder continues the stream at BEST; the setting is fixed once a frame is
    written; and BEST codes the inter frames differently from REALTIME"""
    from alfalfa_b200 import Context, Decoder, Encoder, LogicError, capi
    w, h, qi = 176, 144, 44
    frames = [synth(w, h, t) for t in range(5)]
    ctx = Context(w, h, max_frames=48)
    enc = Encoder(ctx, quality="best")
    clone_before = enc.copy()  # a copy made before the first frame may still change its setting ...
    clone_before.set_quality("realtime")
    clone_before.set_quality("best")
    dec = Decoder(ctx)
    od = O.OracleDecoder(w, h)
    best = []
    for t in range(4):
        blob = enc.encode_with_quantizer(*frames[t], qi)
        best.append(blob)
        want = od.decode(blob)
        rec = enc.reconstruction()
        for g, w_ in zip(rec.planes(), want["planes"]):
            assert np.array_equal(g, w_), "frame %d: the oracle's decode differs from the reconstruction" % t
        rec.release()
        dec.get_frame_output(blob)[1].release()
        assert enc.export_decoder() == dec
        st = enc.stats()
        assert st["y_ac_qi"] == qi and st["loop_filter_level"] == od.parsed().desc.loop_filter_level
        with pytest.raises(LogicError):
            enc.set_quality("realtime")
    assert clone_before.encode_with_quantizer(*frames[0], qi) == best[0]
    with pytest.raises(LogicError):
        enc.set_quality("fast")
    fresh = Encoder(ctx)
    for code in (-1, 2):
        assert fresh.L.vp8gpu_encoder_set_quality(fresh.h, code) == capi.ERR_LOGIC
    # REALTIME on the same frames: the same key frame, other inter frames
    realtime = [fresh.encode_with_quantizer(*f, qi) for f in frames[:4]]
    assert realtime[0] == best[0] and realtime[1:] != best[1:]
    # a copy continues at BEST (and cannot change it): the same next frame as the original's
    a = enc.copy()
    with pytest.raises(LogicError):
        a.set_quality("realtime")
    nxt = a.encode_with_quantizer(*frames[4], qi)
    assert nxt == enc.copy().encode_with_quantizer(*frames[4], qi)
    # Encoder( const Decoder &, two_pass, BEST_QUALITY ), and the same through set_quality
    cont = Encoder.from_decoder(ctx, dec, quality="best")
    cont2 = Encoder.from_decoder(ctx, dec)
    cont2.set_quality("best")
    blob = cont.encode_with_quantizer(*frames[4], qi)
    assert blob[0] & 1 and blob == cont2.encode_with_quantizer(*frames[4], qi)
    dec.get_frame_output(blob)[1].release()
    assert cont.export_decoder() == dec and cont2.export_decoder() == dec
    st = cont.stats()
    assert st["y_ac_qi"] == qi and st["loop_filter_level"] >= 0
    del enc, clone_before, fresh, a, cont, cont2, dec
    ctx.close()
