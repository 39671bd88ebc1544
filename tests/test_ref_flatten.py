"""The reference's own parser in front of the product's seam (INTEGRATION.md B, SURVEY.md 8b "narrowest seam").
oracle/_ref/ref_flatten is built from the UNMODIFIED reference front end plus flatten() (oracle/ref_tools/
ref_flatten.cc): reference Frame object -> flat records of include/vp8gpu.h.
CPU part: on every golden vector and the feature-complete stream those records equal, byte for byte, what the
product's front end (vp8gpu_parse_frame) emits -- two independent parsers, one record format.
GPU part: ref_flatten decode drives vp8gpu_decode_parsed with the reference's parse and Frame::copy_to on
device handles; its output must hash to the vector's name like the reference's decode-to-stdout."""
import ctypes as C
import hashlib
import os
import subprocess

import pytest

import oracle_lib as O
import reference_outputs as R
from alfalfa_b200 import capi
from conftest import GOLDEN_DIR, golden_vectors

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TOOL = os.path.join(ROOT, "oracle", "_ref", "ref_flatten")
needs_tool = pytest.mark.skipif(not os.path.exists(TOOL), reason="oracle/_ref/ref_flatten not built (make -C oracle ref)")


def _product_records(path):
    L = capi.lib()
    w, h, frames = O.read_ivf(open(path, "rb").read())
    st, pf = C.c_void_p(), C.c_void_p()
    capi.check(L.vp8gpu_state_create(w, h, C.byref(st)))
    capi.check(L.vp8gpu_parsed_create(C.byref(pf)))
    out, started = [], False
    for f in frames:
        if not started and (f[0] & 1):
            continue
        started = True
        assert L.vp8gpu_parse_frame(st, f, len(f), pf) == 0
        d = L.vp8gpu_parsed_desc(pf).contents
        n = d.mb_cols * d.mb_rows
        out.append(bytes(d) + C.string_at(L.vp8gpu_parsed_mbs(pf), n * 32) +
                   (C.string_at(L.vp8gpu_parsed_tokens(pf), d.n_tokens * 4) if d.n_tokens else b"") +
                   (C.string_at(L.vp8gpu_parsed_split(pf), d.n_split * 64) if d.n_split else b""))
    L.vp8gpu_state_destroy(st)
    L.vp8gpu_parsed_destroy(pf)
    return out


def _check_records(path):
    ours = _product_records(path)
    if not os.path.exists(TOOL):  # the digest of the reference's records, stored where the tool was built
        k = R.key("ref_flatten records", open(path, "rb").read())
        assert R.digest(b"".join(ours)) == R.stored(k)[0], "the product front end's records differ from the reference's"
        return len(ours)
    theirs = subprocess.run([TOOL, "records", path], stdout=subprocess.PIPE, check=True).stdout
    R.check(R.key("ref_flatten records", open(path, "rb").read()), [theirs])
    pos = 0
    for i, rec in enumerate(ours):
        got = theirs[pos:pos + len(rec)]
        if got != rec:
            k = next(j for j in range(min(len(got), len(rec))) if got[j] != rec[j]) if len(got) == len(rec) else -1
            raise AssertionError("frame %d: flattened reference records differ from the product front end's at byte %d" % (i, k))
        pos += len(rec)
    assert pos == len(theirs)
    return len(ours)


@pytest.mark.parametrize("name", golden_vectors())
def test_flattened_reference_frames_equal_the_product_front_end(name):
    assert _check_records(os.path.join(GOLDEN_DIR, name)) >= 1


def test_flatten_on_the_feature_complete_stream():
    assert _check_records(os.path.join(ROOT, "bench_data", "features1080p_12f.ivf")) == 12


@needs_tool
@pytest.mark.gpu
def test_reference_parser_in_front_of_the_seam_reproduces_the_golden_sha1s(tmp_path):
    """one process per frame size: the reference's frame pool allows a single size per process"""
    lib = os.path.join(ROOT, "alfalfa_b200", "libvp8gpu.so")
    groups = {}
    for name in golden_vectors():
        w, h, _ = O.read_ivf(open(os.path.join(GOLDEN_DIR, name), "rb").read())
        groups.setdefault((w, h), []).append(name)
    bad = []
    for (w, h), group in groups.items():
        out = subprocess.run([TOOL, "decode", lib, "--out", str(tmp_path)] + [os.path.join(GOLDEN_DIR, n) for n in group],
                             stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=600)
        if out.returncode != 0:
            bad.append((w, h, out.returncode, out.stderr.decode()[-200:]))
            continue
        for n in group:
            if hashlib.sha1(open(os.path.join(str(tmp_path), n + ".yuv"), "rb").read()).hexdigest() != n:
                bad.append(n)
    assert not bad, bad
