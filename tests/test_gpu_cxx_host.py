"""C++ programs written against the host mirror alfalfa_b200/host/alfalfa_gpu.hh (the reference's Decoder /
Encoder class surface over the C ABI), compiled with g++ and run on the GPU box:
  tests/cxx/decode_to_stdout.cc  the reference's src/tests/decode-to-stdout.cc shape; SHA-1 of its output
                                 must equal the vector's name (tests/decoding.test:14-15) for all 53 vectors
  tests/cxx/encoder_copies.cc    salsify-sender.cc:492-518: an Encoder copied twice per frame, both copies
                                 encoding concurrently, export_decoder / Encoder( Decoder ) round trip
  tests/cxx/reencode_chunk.cc    frontend/xc-enc.cc:262-327 ("xc-enc --reencode"): Encoder( Decoder ).reencode over a
                                 prediction stream; output equal to the reference's own Encoder::reencode"""
import hashlib
import os
import subprocess

import pytest

from conftest import GOLDEN_DIR, golden_vectors

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# the library the programs link: the product's, or -- when tests/test_simt_emulation.py re-runs this file on the CPU --
# the SIMT-emulated build of the same sources (same C ABI)
LIB = os.environ.get("VP8GPU_LIB", os.path.join(ROOT, "alfalfa_b200", "libvp8gpu.so"))
LIBDIR = os.path.dirname(LIB)


def _build(tmp_path_factory, name):
    out = str(tmp_path_factory.mktemp("cxx") / name)
    subprocess.check_call(["g++", "-std=c++14", "-O2", "-Wall", "-Wextra", "-pthread", os.path.join(ROOT, "tests", "cxx", name + ".cc"),
                           "-o", out, "-L" + LIBDIR, "-l:" + os.path.basename(LIB), "-Wl,-rpath," + LIBDIR])
    return out


@pytest.fixture(scope="module")
def decode_to_stdout(tmp_path_factory):
    return _build(tmp_path_factory, "decode_to_stdout")


def test_cxx_programs_compile(tmp_path_factory):
    """CPU part: both programs compile and link against the library (no device needed)"""
    _build(tmp_path_factory, "decode_to_stdout")
    _build(tmp_path_factory, "encoder_copies")
    _build(tmp_path_factory, "reencode_chunk")


def _by_size(names):
    import oracle_lib as O
    groups = {}
    for name in names:
        w, h, _ = O.read_ivf(open(os.path.join(GOLDEN_DIR, name), "rb").read())
        groups.setdefault((w, h), []).append(name)
    return groups


@pytest.mark.gpu
@pytest.mark.parametrize("device_tokens", [0, 1])
def test_cxx_decoder_reproduces_the_golden_sha1s(decode_to_stdout, device_tokens, tmp_path):
    """one process per frame size (one Context), a fresh Decoder per vector"""
    names = [n for n in golden_vectors() if not device_tokens or n.startswith(("0", "4", "f"))]
    bad = []
    for (w, h), group in _by_size(names).items():
        out = subprocess.run([decode_to_stdout, "--out", str(tmp_path), str(device_tokens)] +
                             [os.path.join(GOLDEN_DIR, n) for n in group], stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=600)
        if out.returncode != 0:
            bad.append((w, h, out.returncode, out.stderr.decode()[-200:]))
            continue
        for n in group:
            if hashlib.sha1(open(os.path.join(str(tmp_path), n + ".yuv"), "rb").read()).hexdigest() != n:
                bad.append(n)
    assert not bad, bad


@pytest.mark.gpu
def test_cxx_encoder_copies_encode_concurrently(tmp_path_factory):
    exe = _build(tmp_path_factory, "encoder_copies")
    out = subprocess.run([exe], stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=600)
    assert out.returncode == 0 and out.stdout.decode().startswith("ok"), out.stderr.decode()[-500:]


@pytest.mark.gpu
@pytest.mark.parametrize("extra_frame_chunk", [0, 1])
def test_cxx_reencode_equals_the_reference(tmp_path_factory, tmp_path, extra_frame_chunk):
    """the xc-enc --reencode shape on the mirror against oracle/_ref/ref_reencode: same emitted frames"""
    import numpy as np
    import oracle_lib as O
    import test_gpu_reencode as R
    from reference_outputs import digests
    exe = _build(tmp_path_factory, "reencode_chunk")
    w, h, n = 176, 144, 4
    targets, pred, state = R.make_case(w, h, n, qi_a=36, qi_b=60)
    want = R.reference_reencode(w, h, targets, pred, state, 0.75, bool(extra_frame_chunk))
    raw, pivf, sbin, out = (str(tmp_path / x) for x in ("t.yuv", "p.ivf", "s.bin", "o.ivf"))
    with open(raw, "wb") as f:
        for planes in targets:
            for p in planes:
                f.write(np.ascontiguousarray(p).tobytes())
    open(pivf, "wb").write(R.ivf_bytes(w, h, pred))
    open(sbin, "wb").write(state)
    r = subprocess.run([exe, out, str(w), str(h), raw, pivf, sbin, "0.75", str(extra_frame_chunk)], stdout=subprocess.PIPE,
                       stderr=subprocess.PIPE, timeout=600)
    assert r.returncode == 0 and r.stdout.decode().startswith("ok"), r.stderr.decode()[-500:]
    _, _, got = O.read_ivf(open(out, "rb").read())
    assert digests(got) == want
