"""DecoderState / Decoder serialisation in the reference's tag-length-value format
(decoder/enc_state_serializer.hh:43-190, decoder.cc:54-81, 177-330, probability_tables.cc:126-158).
CPU part: after N frames of a stream the product front end's state, serialised by vp8gpu_state_serialize, is
byte-identical to the DECODER_STATE record inside the unmodified reference's Decoder::serialize output
(oracle/_ref/ref_dump state), on vectors with and without segmentation / loop-filter adjustments; the blob
deserialises to an equal state.
GPU part: the whole Decoder blob (state + LAST raster) equals the reference's byte for byte; a Decoder
deserialised from the REFERENCE's blob continues the stream bit-exactly, and the reference resumes from OUR blob
(ref_dump resume) with the reference decode's output."""
import ctypes as C
import os
import subprocess
import tempfile

import pytest

import oracle_lib as O
import reference_outputs as R
from alfalfa_b200 import capi
from conftest import GOLDEN_DIR, golden_vectors

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FEATURES = os.path.join(ROOT, "bench_data", "features1080p_12f.ivf")


def _ref_blob(path, n):
    return subprocess.run([R.tool("ref_dump"), "state", path, str(n)], stdout=subprocess.PIPE, check=True).stdout


def _state_record(blob):
    assert blob[0] == 11 and int.from_bytes(blob[1:5], "little") == len(blob) - 5      # DECODER
    assert blob[5] == 4                                                                # DECODER_STATE
    n = int.from_bytes(blob[6:10], "little")
    return blob[5:5 + 5 + n]


def _ref_state_record(path, n):
    """digest of the DECODER_STATE record of the reference's Decoder::serialize after n frames of `path`"""
    k = R.key("ref_dump state record", open(path, "rb").read(), n)
    return R.expected(k, (lambda: [_state_record(_ref_blob(path, n))]) if R.tool("ref_dump") else None)[0]


def _ref_blob_digest(path, n):
    """digest of the reference's whole Decoder::serialize blob (state + LAST raster) after n frames of `path`"""
    k = R.key("ref_dump state", open(path, "rb").read(), n)
    return R.expected(k, (lambda: [_ref_blob(path, n)]) if R.tool("ref_dump") else None)[0]


def _ref_resume_digest(blob, path, n):
    """digest of what the reference shows after resuming from `blob` at frame n of `path` (ref_dump resume)"""
    def run():
        with tempfile.NamedTemporaryFile(suffix=".state") as tf:
            tf.write(blob)
            tf.flush()
            return [subprocess.run([R.tool("ref_dump"), "resume", tf.name, path, str(n)], stdout=subprocess.PIPE, check=True).stdout]
    return R.expected(R.key("ref_dump resume", blob, open(path, "rb").read(), n), run if R.tool("ref_dump") else None)[0]


def _product_state_blob(path, n):
    L = capi.lib()
    w, h, frames = O.read_ivf(open(path, "rb").read())
    st, pf = C.c_void_p(), C.c_void_p()
    capi.check(L.vp8gpu_state_create(w, h, C.byref(st)))
    capi.check(L.vp8gpu_parsed_create(C.byref(pf)))
    for f in frames[:n]:
        assert L.vp8gpu_parse_frame(st, f, len(f), pf) == 0
    size = L.vp8gpu_state_serialize(st, None, 0)
    buf = (C.c_uint8 * size)()
    assert L.vp8gpu_state_serialize(st, buf, size) == size
    blob = bytes(buf)
    st2 = C.c_void_p()
    assert L.vp8gpu_state_deserialize(blob, len(blob), C.byref(st2)) == 0
    assert L.vp8gpu_state_equal(st, st2) == 1 and L.vp8gpu_state_hash(st) == L.vp8gpu_state_hash(st2)
    for s in (st, st2):
        L.vp8gpu_state_destroy(s)
    L.vp8gpu_parsed_destroy(pf)
    return blob


@pytest.mark.parametrize("name", golden_vectors())
def test_state_record_equals_the_reference(name):
    path = os.path.join(GOLDEN_DIR, name)
    _, _, frames = O.read_ivf(open(path, "rb").read())
    if frames[0][0] & 1:
        pytest.skip("vector does not start with a key frame")
    for n in sorted({1, min(len(frames), 7), min(len(frames), 29)}):
        assert R.digest(_product_state_blob(path, n)) == _ref_state_record(path, n), "after %d frames" % n


def test_state_record_on_the_feature_stream_with_segmentation_and_filter_deltas():
    kinds = set()
    for n in (1, 3, 5, 8, 12):
        ours = _product_state_blob(FEATURES, n)
        assert R.digest(ours) == _ref_state_record(FEATURES, n)
        body = ours[9 + 5 + 1101:]
        kinds.add((body[0], ours[-14] if body[0] == 6 else None))
    assert any(k[0] == 6 for k in kinds), "no position with segmentation enabled was covered"


def test_state_deserialize_rejects_garbage():
    L = capi.lib()
    st = C.c_void_p()
    assert L.vp8gpu_state_deserialize(b"V8S\x01" + bytes(2000), 2004, C.byref(st)) != 0
    good = _product_state_blob(os.path.join(GOLDEN_DIR, golden_vectors()[0]), 1)
    assert L.vp8gpu_state_deserialize(good[:-1], len(good) - 1, C.byref(st)) != 0
    bad = bytearray(good)
    bad[9 + 5 - 5] ^= 0xFF
    assert L.vp8gpu_state_deserialize(bytes(bad[:9]) + b"\x07" + bytes(bad[10:]), len(bad), C.byref(st)) != 0


@pytest.mark.gpu
@pytest.mark.parametrize("path,n", [(os.path.join(GOLDEN_DIR, "0b546dad90ddefea5085c7751b5fa2f117630b1c"), 9),
                                     (os.path.join(GOLDEN_DIR, "2a4c049c2f8e3a19ee39ffd7074cecd68006a101"), 20)])
def test_decoder_blob_equals_the_reference_and_both_sides_resume_from_it(path, n):
    from alfalfa_b200 import Context, Decoder
    L = capi.lib()
    data = open(path, "rb").read()
    w, h, frames = O.read_ivf(data)
    ctx = Context(w, h, max_frames=32)
    dec = Decoder(ctx)
    for f in frames[:n]:
        _, r = dec.get_frame_output(f)
        r.release()
    size = C.c_size_t(0)
    assert L.vp8gpu_decoder_serialize(dec.h, None, 0, C.byref(size)) == capi.ERR_NOMEM
    ours = dec.serialize()
    assert len(ours) == size.value
    # golden / alternative are not part of the format: the reference blob only carries LAST as well
    assert R.digest(ours) == _ref_blob_digest(path, n)
    theirs = _ref_blob(path, n) if R.tool("ref_dump") else ours  # (byte-equal, by the digest above)
    # (a) the product resumes from the REFERENCE's blob
    resumed = Decoder.deserialize(ctx, theirs)
    # the truth for "resume with golden = alternative = last": the reference itself, from its own blob
    want = _ref_resume_digest(ours, path, n)
    got = b""
    for f in frames[n:]:
        shown, r = resumed.get_frame_output(f)
        if shown:
            got += r.display_bytes()
        r.release()
    # (b) ... and that run of the reference read OUR blob: both continuations agree
    assert R.digest(got) == want
    del dec, resumed
    ctx.close()
