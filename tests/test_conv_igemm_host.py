"""Host-side checks of the tcgen05 implicit-GEMM convolution (csrc/conv_igemm.cu, csrc/conv_igemm_host.cu) that need
no GPU: its shape query, the argument validation of the C entry point and the ops wrapper, and where its tensor-core
code lives (libe2e_asr_b200_tc.so: tcgen05 only, no legacy mma.sync / wgmma path)."""
import ctypes
import re
import shutil
import subprocess

import pytest
import torch


def test_supported_query():
    from e2e_asr_pytorch_b200 import _lib, ops
    lib = _lib.load()
    for c, cout in ((128, 128), (128, 256), (256, 256), (256, 128)):
        assert lib.e2e_conv3x3_igemm_supported(c, cout) == 1
        assert ops.conv3x3_igemm_supported(c, cout)
    for c, cout in ((4, 128), (64, 128), (128, 64), (192, 256), (512, 256), (128, 384), (0, 128)):
        assert lib.e2e_conv3x3_igemm_supported(c, cout) == 0


def test_argument_validation_needs_no_device():
    from e2e_asr_pytorch_b200 import _lib
    lib = _lib.load()
    fake = ctypes.c_void_p(256)                      # a non-null, aligned "device pointer" that is never dereferenced
    odd = ctypes.c_void_p(260)
    ok = lambda *a: lib.e2e_conv3x3_igemm(*a)
    assert ok(None, fake, 1, 4, 4, 128, fake, fake, 128, 1, fake, None) == -1                 # no input
    assert b"e2e_conv3x3_igemm" in lib.e2e_last_error()
    assert ok(fake, fake, 1, 4, 4, 128, fake, None, 128, 1, fake, None) == -1                 # the epilogue needs a bias
    assert ok(fake, fake, 1, 4, 4, 128, fake, fake, 128, 3, fake, None) == -1                 # no such epilogue
    assert ok(fake, fake, 0, 4, 4, 128, fake, fake, 128, 1, fake, None) == -1                 # empty batch
    assert ok(fake, fake, 1, 4, 4, 64, fake, fake, 128, 1, fake, None) == -3                  # shape refused by the query
    assert ok(fake, fake, 1, 4, 4, 128, fake, fake, 192, 1, fake, None) == -3
    assert ok(odd, fake, 1, 4, 4, 128, fake, fake, 128, 1, fake, None) == -1                  # misaligned input
    assert b"misaligned" in lib.e2e_last_error()


def test_wrapper_has_no_cpu_path():
    from e2e_asr_pytorch_b200 import _lib, ops
    x = torch.zeros(1, 4, 4, 128)
    w = torch.zeros(3, 128, 9 * 128, dtype=torch.bfloat16)
    with pytest.raises(_lib.E2EError):
        ops.conv3x3_igemm(x, torch.ones(1, dtype=torch.int32), w, torch.zeros(128), "relu")


def test_tensor_core_kernels_are_tcgen05_in_their_own_library():
    """The implicit-GEMM convolution's MMAs are tcgen05 (UTCHMMA, fed by UTMALDG, read back with LDTM) and live in
    libe2e_asr_b200_tc.so, which the main library links against; neither library has a legacy warp-level HMMA
    (mma.sync) or Hopper HGMMA (wgmma), matched as whole mnemonics."""
    import os
    from e2e_asr_pytorch_b200 import build
    if shutil.which("cuobjdump") is None:
        pytest.skip("cuobjdump not available")
    main = build.build()
    tc = os.path.join(os.path.dirname(main), "libe2e_asr_b200_tc.so")
    ldd = subprocess.run(["readelf", "-d", main], capture_output=True, text=True).stdout if shutil.which("readelf") else ""
    if ldd:
        assert "libe2e_asr_b200_tc.so" in ldd and "$ORIGIN" in ldd
    sass_tc = subprocess.run(["cuobjdump", "-sass", tc], capture_output=True, text=True).stdout
    sass_main = subprocess.run(["cuobjdump", "-sass", main], capture_output=True, text=True).stdout
    assert "sm_100a" in sass_tc and "conv3x3_igemm_kernel" in sass_tc
    for m in ("UTCHMMA", "UTCBAR", "LDTM", "UTMALDG"):
        assert re.search(r"\b%s\b" % m, sass_tc), m
    for sass in (sass_tc, sass_main):
        assert not re.search(r"\bHMMA\b", sass) and not re.search(r"\bHGMMA\b", sass)
