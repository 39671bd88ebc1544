"""Re-encoding on the GPU (SURVEY.md 8 row f3): Encoder::reencode / update_residues (encoder/reencode.cc) against the
UNMODIFIED reference's Encoder::reencode (oracle/_ref/ref_reencode, driven like frontend/xc-enc.cc:262-327).

The ExCamera situation: a chunk was coded on its own (it starts with a key frame); a receiver, however, arrives at the
chunk in the state the PREVIOUS chunk left it in.  Re-encoding keeps the chunk's modes and vectors and recomputes
its residues against the references the receiver really has.  Both sides get the same serialized Decoder (the
reference's EncoderStateSerializer blob), the same prediction stream and the same target rasters; the emitted frames
must be equal byte for byte, and a decoder resumed from the blob must decode them to the same pictures.

This file also runs on the CPU under the SIMT emulator (tests/test_simt_emulation.py), at the small size only."""
import os
import subprocess
import tempfile

import numpy as np
import pytest

import oracle_lib as O
import reference_outputs as R
from test_gpu_encoder import ROOT, reference_encode, synth

pytestmark = pytest.mark.gpu
EMULATED = bool(os.environ.get("VP8GPU_SIMT_EMULATED"))
SIZES = [(176, 144)] if EMULATED else [(176, 144), (640, 360)]


def ivf_bytes(w, h, chunks):
    from alfalfa_b200 import write_ivf
    return write_ivf(w, h, chunks)


def reference_reencode(w, h, targets, pred_chunks, state_blob, kf_q_weight, extra_frame_chunk):
    """oracle/_ref/ref_reencode: the reference's Encoder::reencode; returns the digests (reference_outputs.digest) of
    the emitted frames"""
    def run():
        with tempfile.TemporaryDirectory() as d:
            raw, pred, state, out = (os.path.join(d, n) for n in ("t.yuv", "p.ivf", "s.bin", "o.ivf"))
            with open(raw, "wb") as f:
                for planes in targets:
                    for p in planes:
                        f.write(np.ascontiguousarray(p).tobytes())
            open(pred, "wb").write(ivf_bytes(w, h, pred_chunks))
            open(state, "wb").write(state_blob)
            r = subprocess.run([R.tool("ref_reencode"), out, str(w), str(h), raw, pred, state, repr(kf_q_weight),
                                str(int(extra_frame_chunk))], capture_output=True, text=True)
            assert r.returncode == 0, r.stderr[-400:]
            return O.read_ivf(open(out, "rb").read())[2]
    k = R.key("ref_reencode", w, h, targets, pred_chunks, state_blob, kf_q_weight, bool(extra_frame_chunk))
    return R.expected(k, run if R.tool("ref_reencode") else None)


def reference_state_after(w, h, chunks, n):
    """Decoder::serialize of the reference decoder after n frames (ref_dump state).  Where the reference is not built,
    this library's Decoder::serialize, which must have the digest stored for the reference's blob."""
    k = R.key("ref_dump state", w, h, chunks[:n])
    if R.tool("ref_dump") is None:
        from alfalfa_b200 import Context, Decoder
        ctx = Context(w, h, max_frames=16)
        dec = Decoder(ctx)
        for c in chunks[:n]:
            dec.get_frame_output(c)[1].release()
        blob = dec.serialize()
        del dec
        ctx.close()
        assert R.digest(blob) == R.stored(k)[0], "Decoder::serialize differs from the reference's blob"
        return blob
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "a.ivf")
        open(path, "wb").write(ivf_bytes(w, h, chunks))
        r = subprocess.run([R.tool("ref_dump"), "state", path, str(n)], capture_output=True)
        assert r.returncode == 0, r.stderr[-400:]
        return R.check(k, [r.stdout])[0]


def make_case(w, h, n, qi_a, qi_b):
    """previous chunk = frames 0..n (ends with frame n coded as an INTER frame); this chunk = frames n..2n-1 coded on
    its own (frame n is its key frame).  Extra-frame re-encoding starts at this chunk's second frame."""
    frames = [synth(w, h, t) for t in range(2 * n)]
    prev = reference_encode(frames[:n + 1], w, h, qi=qi_a)
    pred = reference_encode(frames[n:], w, h, qi=qi_b)
    state = reference_state_after(w, h, prev, n + 1)
    return frames[n:], pred, state


def product_reencode(w, h, targets, pred_chunks, state_blob, kf_q_weight, extra_frame_chunk, timeout=300, env=None):
    """the product's Encoder::reencode in a child process (tests/reencode_worker.py) under a timeout: returns
    (emitted frames, receiver-in-step flag)"""
    import pickle
    import sys
    with tempfile.TemporaryDirectory() as d:
        fin, fout = os.path.join(d, "in.pickle"), os.path.join(d, "out.pickle")
        pickle.dump(dict(w=w, h=h, targets=[tuple(np.ascontiguousarray(p) for p in t) for t in targets], pred=list(pred_chunks),
                         state=bytes(state_blob), kf_q_weight=kf_q_weight, extra_frame_chunk=bool(extra_frame_chunk)), open(fin, "wb"))
        r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "reencode_worker.py"), fin, fout], capture_output=True, text=True,
                           timeout=timeout, env=dict(os.environ, **(env or {})))
        assert r.returncode == 0, (r.stdout + r.stderr)[-1500:]
        out = pickle.load(open(fout, "rb"))
    return out["frames"], out["in_step"]


def test_whole_chunk_the_same_with_the_shortcuts_off():
    """VP8GPU_ENC_SPECULATE=0: the loop-filter trials one by one and the decode of every written frame through the
    full parse instead of the token lists it was written from -- the same bytes, the receiver still in step"""
    w, h = SIZES[-1]
    n = 4
    targets, pred, state = make_case(w, h, n, qi_a=40, qi_b=64)
    want = reference_reencode(w, h, targets, pred, state, 0.75, False)
    got, in_step = product_reencode(w, h, targets, pred, state, 0.75, False, env={"VP8GPU_ENC_SPECULATE": "0"})
    assert R.digests(got) == want and in_step


@pytest.mark.parametrize("size", SIZES)
@pytest.mark.parametrize("kf_q_weight", [1.0, 0.75])
def test_extra_frame_chunk_is_reencoded_byte_for_byte_like_the_reference(size, kf_q_weight):
    """Encoder::reencode options 2 and 4 (reencode.cc:353-373): update_residues with a blended quantiser for the first
    frame, with the frame's own quantiser afterwards, all references refreshed by the last one"""
    w, h = size
    n = 4
    targets, pred, state = make_case(w, h, n, qi_a=40, qi_b=56)
    want = reference_reencode(w, h, targets, pred, state, kf_q_weight, True)
    got, in_step = product_reencode(w, h, targets, pred, state, kf_q_weight, True)
    assert len(got) == len(want) == n - 1
    for i, (a, b) in enumerate(zip(got, want)):
        assert R.digest(a) == b, "frame %d: %d vs %d bytes" % (i + 1, len(a), b[0])
    # and the Encoder moved the way a receiver moves: a decoder resumed from the blob that decodes the emitted
    # frames ends up equal to export_decoder()
    assert in_step


@pytest.mark.parametrize("size", SIZES)
@pytest.mark.parametrize("kf_q_weight", [1.0, 0.5])
def test_whole_chunk_is_reencoded_byte_for_byte_like_the_reference(size, kf_q_weight):
    """Encoder::reencode options 1 and 4 (reencode.cc:336-351, 366-372): the chunk's key frame becomes an inter frame
    predicted from the receiver's LAST (reencode_as_interframe: the full decision loop, quantiser blended with the
    next frame's), the other frames keep their decisions and get new residues"""
    w, h = size
    n = 4
    targets, pred, state = make_case(w, h, n, qi_a=40, qi_b=64)
    want = reference_reencode(w, h, targets, pred, state, kf_q_weight, False)
    got, in_step = product_reencode(w, h, targets, pred, state, kf_q_weight, False)
    assert len(got) == len(want) == n
    for i, (a, b) in enumerate(zip(got, want)):
        assert R.digest(a) == b, "frame %d: %d vs %d bytes" % (i, len(a), b[0])
    assert got[0][0] & 1, "the chunk no longer starts with a key frame"
    assert in_step


def test_reencoded_frames_differ_from_the_prediction_frames_but_keep_their_modes():
    """the point of update_residues: same decisions, new residues (the references are another reconstruction)"""
    w, h, n = 176, 144, 3
    targets, pred, state = make_case(w, h, n, qi_a=30, qi_b=60)
    got, _ = product_reencode(w, h, targets, pred, state, 1.0, True)
    from alfalfa_b200 import Context, Decoder
    ctx = Context(w, h, max_frames=24)   # (the comparison below only decodes: kernels with a hardware record)
    a, b = Decoder(ctx), Decoder.deserialize(ctx, state)
    a.get_frame_output(pred[0])
    for new, old in zip(got, pred[1:]):
        assert new != old
        pa, pb = a.parse_frame(old), b.parse_frame(new)
        a.decode_frame(pa), b.decode_frame(pb)
        (ma, _, sa), (mb, _, sb) = pa.arrays(), pb.arrays()
        for key in ("y_mode", "uv_mode", "ref_frame", "mv_x", "mv_y", "b_modes"):
            assert np.array_equal(ma[key], mb[key]), key
        assert np.array_equal(sa, sb)
    ctx.close()


def test_update_residues_argument_errors():
    """LogicError / Unsupported where the reference throws or where the call cannot mean anything (child process, see
    tests/reencode_worker.py)"""
    import sys
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "reencode_worker.py"), "errors"], capture_output=True, text=True,
                       timeout=300)
    assert r.returncode == 0 and "ok" in r.stdout, (r.stdout + r.stderr)[-1500:]


def _decoded_targets(w, h, chunks):
    """the prediction stream's own pictures (every frame, shown or not) as targets: ExCamera re-encodes a chunk
    towards what the chunk looked like when it was coded on its own"""
    from alfalfa_b200 import Context, Decoder
    ctx = Context(w, h, max_frames=16)
    d = Decoder(ctx)
    cw, ch = (w + 1) // 2, (h + 1) // 2
    out = []
    for c in chunks:
        _, r = d.get_frame_output(c)
        b = np.frombuffer(r.display_bytes(), np.uint8)
        out.append((b[:w * h].reshape(h, w), b[w * h:w * h + cw * ch].reshape(ch, cw), b[w * h + cw * ch:].reshape(ch, cw)))
    ctx.close()
    return out


def _golden(name):
    from conftest import GOLDEN_DIR
    return O.read_ivf(open(os.path.join(GOLDEN_DIR, name), "rb").read())


# prediction streams written by libvpx (the reference's own test vectors): SPLITMV with every layout, golden and
# altref prediction with sign bias, B_PRED and 16x16 intra macroblocks inside inter frames, loop-filter deltas,
# segmentation without a map update, several token partitions, hidden frames, odd sizes.
# (previous chunk, this chunk, frames)
VECTOR_CASES = [
    ("04b68b0a642d8285303d2b8884fc374e09d28ae9", "07b5eb1e9741d90027c46166eaaff566c6bf934f", 20),
    ("04b68b0a642d8285303d2b8884fc374e09d28ae9", "4fca93f3", 28),
    ("9038efed", "7d865ecf", 29),
    ("7d865ecf", "9038efed", 20),
    ("07b5eb1e9741d90027c46166eaaff566c6bf934f", "a4dace04", 14),
    ("a4dace04", "ced8ea72", 30),
    ("a4dace04", "df225756", 30),
    ("0ccf971d", "353ee97f", 15),
    ("353ee97f", "a61782d0", 15),
    ("a61782d0", "dbdd0703", 13),
    ("d1e7b447", "de0dc731", 24),
]


def _full_name(prefix):
    from conftest import golden_vectors
    hits = [n for n in golden_vectors() if n.startswith(prefix)]
    assert len(hits) == 1, prefix
    return hits[0]


@pytest.mark.parametrize("prev,this,nframes", VECTOR_CASES)
def test_update_residues_on_libvpx_prediction_streams(prev, this, nframes):
    pw, ph, prev_chunks = _golden(_full_name(prev))
    w, h, chunks = _golden(_full_name(this))
    assert (pw, ph) == (w, h)
    chunks = chunks[:nframes]
    if EMULATED:
        chunks = chunks[:12]
    state = reference_state_after(w, h, prev_chunks, len(prev_chunks))
    targets = _decoded_targets(w, h, chunks)
    want = reference_reencode(w, h, targets, chunks, state, 0.75, True)
    got, in_step = product_reencode(w, h, targets, chunks, state, 0.75, True)
    assert len(got) == len(want) == len(chunks) - 1
    for i, (a, b) in enumerate(zip(got, want)):
        assert R.digest(a) == b, "frame %d: %d vs %d bytes" % (i + 1, len(a), b[0])
    assert in_step


@pytest.mark.parametrize("prev", ["07b5eb1e", "4fca93f3", "a4dace04", "ced8ea72", "d4e9f670", "df225756"])
def test_whole_chunk_after_a_libvpx_stream(prev):
    """options 1 + 4 when the receiver's state comes from a libvpx stream: updated motion-vector and mode
    probabilities (the rate tables of the decision loop are rebuilt from them, Costs::fill_mv_component_costs
    reencode.cc:82-85; macroblock headers are coded with them), loop-filter adjustments, golden / altref that differ
    from LAST"""
    w, h, prev_chunks = _golden(_full_name(prev))
    n = 4
    frames = [synth(w, h, t) for t in range(n)]
    pred = reference_encode(frames, w, h, qi=60)
    state = reference_state_after(w, h, prev_chunks, len(prev_chunks))
    want = reference_reencode(w, h, frames, pred, state, 0.75, False)
    got, in_step = product_reencode(w, h, frames, pred, state, 0.75, False)
    assert R.digests(got) == want and in_step
