"""The BEST_QUALITY encoder (tests/test_gpu_encoder_best_quality.py) under the SIMT emulator, in both thread orders:
k_enc_rd with the B_PRED trial and the motion search at every inter-frame macroblock, the sub-block contexts inter
macroblocks hand on, the searches that start from scratch every frame, and re-encoding at BEST -- byte for byte against
the reference encoder built at BEST (oracle/_ref/ref_encode_best, ref_reencode_best; or their stored digests).  The
1080p case stays on the GPU."""
import pytest

from test_simt_emulation import pytestmark, run_gpu_tests_emulated, simt_lib  # noqa: F401

ARGS = ["tests/test_gpu_encoder_best_quality.py", "-k", "not 1080p"]


def test_best_quality_encoder_emulated(simt_lib):  # noqa: F811
    run_gpu_tests_emulated(simt_lib, ARGS, timeout=1800)


@pytest.mark.parametrize("order", ["reverse"])
def test_best_quality_encoder_reverse_thread_order(simt_lib, order):  # noqa: F811
    """SIMT_ORDER=reverse: a shared-memory hand-over between lanes without its barrier shows in one of the two orders"""
    run_gpu_tests_emulated(simt_lib, ARGS, timeout=1800, env_extra={"SIMT_ORDER": order})
