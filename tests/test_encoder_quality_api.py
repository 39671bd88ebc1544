"""The encoder-quality setting at the boundaries that need no GPU: the header's VP8GPU_QUALITY_* values are the reference
enum's order and the Python binding's, and the C++ mirror offers the reference's constructors
Encoder( w, h, two_pass, quality ) and Encoder( const Decoder &, two_pass, quality ) (encoder.hh:346-351)."""
import os
import re
import subprocess
import tempfile

from alfalfa_b200 import capi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_quality_values_follow_the_reference_enum():
    text = open(os.path.join(ROOT, "include", "vp8gpu.h")).read()
    values = dict((k, int(v)) for k, v in re.findall(r"#define\s+VP8GPU_QUALITY_([A-Z]+)\s+(\d+)", text))
    assert values == {"BEST": 0, "REALTIME": 1}
    assert (capi.QUALITY_BEST, capi.QUALITY_REALTIME) == (0, 1)


def test_cxx_mirror_has_the_reference_constructors():
    src = r'''
#include "alfalfa_b200/host/alfalfa_gpu.hh"
static_assert(alfalfa_gpu::BEST_QUALITY == 0 && alfalfa_gpu::REALTIME_QUALITY == 1, "EncoderQuality order");
int use(const uint8_t* data) {
  alfalfa_gpu::Context ctx(0, 320, 240);
  alfalfa_gpu::Encoder enc(ctx, 320, 240, false, alfalfa_gpu::BEST_QUALITY);
  alfalfa_gpu::Decoder dec(ctx, 320, 240);
  alfalfa_gpu::Encoder cont(dec, true, alfalfa_gpu::REALTIME_QUALITY);
  cont.set_quality(alfalfa_gpu::BEST_QUALITY);
  alfalfa_gpu::SourceFrame sf = {data, data, data, 320, 160};
  return (int)enc.encode_with_quantizer(sf, 40).size() + (int)cont.encode_with_quantizer(sf, 40).size();
}
'''
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "quality.cc")
        open(path, "w").write(src)
        subprocess.check_call(["g++", "-std=c++14", "-Wall", "-Wextra", "-shared", "-fPIC", "-I" + ROOT, path, "-o",
                               os.path.join(d, "q.so"), "-L" + os.path.join(ROOT, "alfalfa_b200"), "-l:libvp8gpu.so"])
