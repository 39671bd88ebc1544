"""The product's own sources under a SIMT emulator (tests/simt): TEST INFRASTRUCTURE for the container without a GPU.

tests/simt/build.sh compiles csrc/*.cu / *.cc with g++ against a stand-in <cuda_runtime.h> in which a kernel launch
runs the kernel's threads as fibers (warp collectives = rendez-vous of 32 fibers, CTAs in launch order, streams
synchronous).  The result, tests/simt/_build/libvp8gpu_simt.so, exports the same C ABI; these tests run the
`-m gpu` parity tests against it in a child process (VP8GPU_LIB), so the kernels' logic and the host orchestration
around them are checked bit-exactly here, before the code ever reaches the B200 -- the GPU run then only has to add
what an emulator cannot show (memory ordering, residency, speed).  The product never loads this library and has
no CPU path: alfalfa_b200/libvp8gpu.so without a CUDA device fails in vp8gpu_ctx_create."""
import os
import shutil
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SIMT_DIR = os.path.join(ROOT, "tests", "simt")
SIMT_LIB = os.path.join(SIMT_DIR, "_build", "libvp8gpu_simt.so")

pytestmark = pytest.mark.skipif(shutil.which("g++") is None or os.uname().machine != "x86_64",
                                reason="the emulator's fiber switch is x86-64 and needs g++")


@pytest.fixture(scope="module")
def simt_lib():
    r = subprocess.run(["sh", os.path.join(SIMT_DIR, "build.sh")], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and os.path.exists(SIMT_LIB), r.stderr[-2000:]
    return SIMT_LIB


def run_gpu_tests_emulated(lib, args, timeout=900, env_extra=None):
    """pytest -m gpu <args> in a child process whose alfalfa_b200.capi binds the emulated library"""
    env = dict(os.environ, VP8GPU_LIB=lib, VP8GPU_SIMT_EMULATED="1")
    env.update(env_extra or {})
    r = subprocess.run([sys.executable, "-m", "pytest", "-x", "-q", "-m", "gpu", "-p", "no:cacheprovider"] + args, cwd=ROOT, env=env,
                       capture_output=True, text=True, timeout=timeout)
    tail = (r.stdout + r.stderr)[-3000:]
    assert r.returncode == 0, tail
    assert " passed" in tail and " failed" not in tail, tail
    return tail


def test_emulated_library_exports_the_c_abi(simt_lib):
    """same symbols as the product library: the emulated build is the same sources, nothing stubbed out"""
    import re
    declared = set(re.findall(r"\b(vp8gpu_[a-z0-9_]+)\s*\(", open(os.path.join(ROOT, "include", "vp8gpu.h")).read()))
    out = subprocess.run(["nm", "-D", "--defined-only", simt_lib], capture_output=True, text=True).stdout
    exported = set(re.findall(r"\b(vp8gpu_[a-z0-9_]+)\b", out))
    assert declared and not (declared - exported), sorted(declared - exported)


def test_golden_vectors_through_emulated_kernels(simt_lib):
    """FilePlayer over the golden vectors (k_inter incl. the TMA path, k_intra_ll, k_loopfilter): SHA-1 == name"""
    run_gpu_tests_emulated(simt_lib, ["tests/test_gpu_parity.py", "-k", "fileplayer and not ff2941"])


@pytest.mark.parametrize("mode", ["legacy", "ll"])
def test_both_wavefront_protocols_emulated(simt_lib, mode):
    """round-1 progress counters and the hand-over messages of both wavefront kernels"""
    run_gpu_tests_emulated(simt_lib, ["tests/test_gpu_parity.py", "-k", "every_frame_matches_oracle or (fileplayer and (0b546dad or a4dace04 or e01c6f92))"],
                           env_extra={"VP8GPU_WAVEFRONT": mode})


def test_stream_decode_and_device_token_decoder_emulated(simt_lib):
    """vp8gpu_decode_ivf with worker / dispatcher threads, host tokens and k_tokens; mid-stream failure unwinding"""
    run_gpu_tests_emulated(simt_lib, ["tests/test_gpu_parity.py", "-k", "not fileplayer and not full_size and not ff2941 and not every_frame"])


def test_reencode_against_the_reference_emulated(simt_lib):
    """Encoder::reencode / update_residues (SURVEY 8 f3): k_reenc_inter / k_reenc_intra + the host orchestration,
    byte for byte against the reference's Encoder::reencode on reference-encoder and libvpx prediction streams"""
    run_gpu_tests_emulated(simt_lib, ["tests/test_gpu_reencode.py"])


def test_encoder_against_the_reference_encoder_emulated(simt_lib):
    """k_enc_rd + the encoder's host side: decisions equal to the unmodified reference encoder's, closed loop,
    target-size search, loop-filter choice, value semantics (the 1080p cases stay on the GPU: minutes here)"""
    run_gpu_tests_emulated(simt_lib, ["tests/test_gpu_encoder.py", "-k", "not rd_parity and not first_inter_frame and not size3"])


def test_cxx_callers_on_the_host_mirror_emulated(simt_lib):
    """C++ programs written against alfalfa_gpu.hh, linked with the emulated library: Salsify's concurrent Encoder
    copies (two host threads launching kernels) and the xc-enc --reencode shape against the reference's output"""
    run_gpu_tests_emulated(simt_lib, ["tests/test_gpu_cxx_host.py", "-k", "encoder_copies or reencode"])


def test_reverse_thread_order_gives_the_same_results(simt_lib):
    """SIMT_ORDER=reverse runs the threads of every CTA last to first: together with the default order this exposes a
    shared-memory hand-over between lanes that lacks its barrier (one of the two orders reads before the write)"""
    rev = {"SIMT_ORDER": "reverse"}
    run_gpu_tests_emulated(simt_lib, ["tests/test_gpu_parity.py", "-k", "every_frame_matches_oracle or (fileplayer and not ff2941 and not 2a4c049c)"],
                           env_extra=rev)
    run_gpu_tests_emulated(simt_lib, ["tests/test_gpu_encoder.py", "-k", "decisions_equal and not size3"], env_extra=rev)
    run_gpu_tests_emulated(simt_lib, ["tests/test_gpu_reencode.py"], env_extra=rev)


def test_no_misaligned_vector_access_in_the_kernels(simt_lib):
    """x86 tolerates a misaligned uint4 / uint2 / uint32 access, the GPU faults on it: the emulated build once more
    under -fsanitize=alignment (tests/simt/build.sh, SIMT_SANITIZE), over the re-encoding path (the kernels without a
    hardware run) and a few decode vectors"""
    ubsan = subprocess.run(["g++", "-print-file-name=libubsan.so"], capture_output=True, text=True).stdout.strip()
    if not os.path.isabs(ubsan) or not os.path.exists(ubsan):
        pytest.skip("libubsan not available")
    r = subprocess.run(["sh", os.path.join(SIMT_DIR, "build.sh")], env=dict(os.environ, SIMT_SANITIZE="alignment"), capture_output=True,
                       text=True, timeout=900)
    san = os.path.join(SIMT_DIR, "_build", "san", "libvp8gpu_simt.so")
    assert r.returncode == 0 and os.path.exists(san), r.stderr[-2000:]
    args = ["tests/test_gpu_parity.py", "-k", "fileplayer and (0b546dad or a4dace04 or e01c6f92 or 8bf4c5bb)"]
    run_gpu_tests_emulated(san, args, env_extra={"LD_PRELOAD": ubsan})
    run_gpu_tests_emulated(san, ["tests/test_gpu_reencode.py"], env_extra={"LD_PRELOAD": ubsan})
    # the encoder's predictor (packed filters on staged windows, word stores into the candidate buffers)
    run_gpu_tests_emulated(san, ["tests/test_gpu_encoder.py", "-k", "(decisions_equal and not size3) or two_pass"], env_extra={"LD_PRELOAD": ubsan})
