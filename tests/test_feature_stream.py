"""Feature-complete synthetic streams (tools/make_feature_stream.py; SURVEY.md 8d "bitstream B"):
1-8 DCT partitions, segmentation, loop-filter and quantiser deltas, golden / altref with sign bias,
buffer copies, hidden frames, persistent probabilities, B_PRED and SPLITMV everywhere.
CPU part: the oracle reproduces the reference decoder's SHA-1 of the committed 1080p clip; the host
front end and the device token logic (CPU build) agree with the oracle's records on fresh streams of
odd sizes.  GPU part: every frame (shown or hidden) and the three references equal the oracle's, with
the DCT partitions decoded on the host and on the device."""
import ctypes as C
import hashlib
import json
import os
import subprocess
import sys
import tempfile

import numpy as np
import pytest

import oracle_lib as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
CLIP = "features1080p_12f.ivf"


def _stream(w, h, frames, seed):
    import make_feature_stream
    return make_feature_stream.make_stream(w, h, frames, seed)


def test_oracle_matches_reference_on_the_1080p_feature_clip():
    want = json.load(open(os.path.join(ROOT, "tests", "golden", "bench_clips.json")))[CLIP]
    out = O.decode_ivf_display(open(os.path.join(ROOT, "bench_data", CLIP), "rb").read())
    assert len(out) == want["bytes"] and hashlib.sha1(out).hexdigest() == want["sha1_of_reference_decode"]


def test_feature_clip_is_reproducible():
    """the committed clip is what the generator writes today (writer + generator are deterministic)"""
    assert _stream(1920, 1080, 12, 2024) == open(os.path.join(ROOT, "bench_data", CLIP), "rb").read()


@pytest.mark.parametrize("w,h,seed", [(176, 144, 1), (175, 143, 2), (33, 17, 3), (16, 16, 4), (640, 368, 5)])
def test_host_front_end_and_device_token_logic_on_feature_streams(w, h, seed):
    from alfalfa_b200 import capi
    L = capi.lib()
    data = _stream(w, h, 8, seed)
    _, _, frames = O.read_ivf(data)
    od = O.OracleDecoder(w, h)
    st, pf = C.c_void_p(), C.c_void_p()
    capi.check(L.vp8gpu_state_create(w, h, C.byref(st)))
    capi.check(L.vp8gpu_parsed_create(C.byref(pf)))
    # CPU build of the k_tokens body next to it
    d = tempfile.mkdtemp()
    so = os.path.join(d, "tokens_host.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", os.path.join(ROOT, "tests", "tokens_host_shim.cc"),
                           os.path.join(ROOT, "alfalfa_b200", "csrc", "parser.cc"), "-o", so])
    T = C.CDLL(so)
    T.th_new.restype = C.c_void_p
    T.th_new.argtypes = [C.c_int, C.c_int]
    T.th_frame.argtypes = [C.c_void_p, C.c_char_p, C.c_size_t, C.c_uint32, C.POINTER(C.c_uint32)]
    T.th_variant.argtypes = [C.c_void_p, C.c_int]
    H = T.th_new(w, h)
    T.th_variant(H, seed & 1)   # one thread per frame / the lock-step state machine
    for i, f in enumerate(frames):
        od.decode(f, want_planes=False)
        op = od.parsed()
        assert L.vp8gpu_parse_frame(st, f, len(f), pf) == 0
        desc = L.vp8gpu_parsed_desc(pf).contents
        assert bytes(desc) == bytes(op.desc), "frame %d desc" % i
        n = desc.mb_cols * desc.mb_rows
        assert C.string_at(L.vp8gpu_parsed_mbs(pf), n * 32) == op.mbs.tobytes(), "frame %d mbs" % i
        if desc.n_tokens:
            assert C.string_at(L.vp8gpu_parsed_tokens(pf), desc.n_tokens * 4) == op.tokens.tobytes(), "frame %d tokens" % i
        if desc.n_split:
            assert C.string_at(L.vp8gpu_parsed_split(pf), desc.n_split * 64) == op.split.tobytes(), "frame %d split" % i
        assert T.th_frame(H, f, len(f), 0, None) == 0, "frame %d: device token logic" % i


@pytest.mark.parametrize("seed", range(100, 124))
def test_many_small_feature_streams_oracle_and_front_end_agree(seed):
    """fuzz: every seed draws its own mix of partitions / segmentation / references / modes; sizes cover
    single-row, single-column and non-multiple-of-16 frames"""
    from alfalfa_b200 import capi
    L = capi.lib()
    w, h = [(16, 16), (48, 16), (16, 80), (50, 34), (96, 64), (130, 98)][seed % 6]
    data = _stream(w, h, 6, seed)
    _, _, frames = O.read_ivf(data)
    od = O.OracleDecoder(w, h)
    st, pf = C.c_void_p(), C.c_void_p()
    capi.check(L.vp8gpu_state_create(w, h, C.byref(st)))
    capi.check(L.vp8gpu_parsed_create(C.byref(pf)))
    for i, f in enumerate(frames):
        od.decode(f, want_planes=False)
        op = od.parsed()
        assert L.vp8gpu_parse_frame(st, f, len(f), pf) == 0
        desc = L.vp8gpu_parsed_desc(pf).contents
        n = desc.mb_cols * desc.mb_rows
        assert bytes(desc) == bytes(op.desc), "frame %d desc" % i
        assert C.string_at(L.vp8gpu_parsed_mbs(pf), n * 32) == op.mbs.tobytes(), "frame %d mbs" % i
        if desc.n_tokens:
            assert C.string_at(L.vp8gpu_parsed_tokens(pf), desc.n_tokens * 4) == op.tokens.tobytes(), "frame %d tokens" % i
    L.vp8gpu_parsed_destroy(pf)
    L.vp8gpu_state_destroy(st)


@pytest.mark.gpu
@pytest.mark.parametrize("device_tokens", [False, True])
@pytest.mark.parametrize("source", ["clip", (175, 143, 7), (640, 368, 8)])
def test_gpu_every_frame_and_reference_matches_oracle(source, device_tokens):
    from alfalfa_b200 import Context, Decoder
    data = (open(os.path.join(ROOT, "bench_data", CLIP), "rb").read() if source == "clip"
            else _stream(source[0], source[1], 10, source[2]))
    w, h, frames = O.read_ivf(data)
    ctx = Context(w, h, max_frames=16)
    dec = Decoder(ctx)
    dec.set_device_tokens(device_tokens)
    od = O.OracleDecoder(w, h)
    for i, f in enumerate(frames):
        want = od.decode(f)
        shown, raster = dec.get_frame_output(f)
        assert shown == want["shown"]
        for g, w_ in zip(raster.planes(), want["planes"]):
            assert np.array_equal(g, w_), "frame %d" % i
        raster.release()
    for k, r in enumerate(dec.get_references()):
        for g, w_ in zip(r.planes(), O.raster_planes(od.L.vp8o_decoder_ref(od.d, k))):
            assert np.array_equal(g, w_), "reference %d" % k
        r.release()
    del dec
    ctx.close()


@pytest.mark.parametrize("seed", range(200, 212))
def test_oracle_equals_the_unmodified_reference_decoder_on_fresh_feature_streams(seed):
    """the oracle is pinned by the 53 golden vectors; here also against the reference decoder itself
    (compiled in place by oracle/Makefile, or its stored output where it is not built) on streams of seeded features"""
    import reference_outputs as R
    w, h = [(64, 48), (176, 144), (50, 34), (320, 96)][seed % 4]
    data = _stream(w, h, 8, seed)

    def run():
        with tempfile.NamedTemporaryFile(suffix=".ivf") as f:
            f.write(data)
            f.flush()
            raw = subprocess.run([R.tool("ref_dump"), "shown", f.name], capture_output=True)
        assert raw.returncode == 0, raw.stderr[-500:]
        return [raw.stdout]
    want = R.expected(R.key("ref_dump shown", data), run if R.tool("ref_dump") else None)[0]
    assert R.digest(O.decode_ivf_display(data)) == want
