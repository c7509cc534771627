"""Drop-in at the reference's HLS-top boundary: the reference's UNCHANGED src/main.cpp and
src/openjpg.cpp (compiled by oracle/build_ref.sh into oracle/_ref/ref_main_on_gpu) running on this
repository's JpegDecodeHW (csrc/ref_shim_hw.cpp -> libhjd.so -> CUDA kernels)."""
import hashlib
import os
import shutil
import subprocess

import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "oracle", "_ref", "ref_main_on_gpu")
LENNA = os.path.join(ROOT, "oracle", "_ref", "data", "Lenna.jpg")


def test_reference_main_runs_on_the_gpu_decode_core(tmp_path, port, hjd):
    if not (os.path.exists(BIN) and os.path.exists(LENNA)):
        pytest.skip("oracle/_ref/ref_main_on_gpu not built: needs a checkout of the original project, which is not part "
                    "of this repository (REF=<checkout> oracle/build_ref.sh)")
    # main.cpp hard-codes ../../../../data/Lenna.jpg and ../../../../data/out.bmp (main.cpp:30-31)
    (tmp_path / "data").mkdir()
    shutil.copy(LENNA, tmp_path / "data" / "Lenna.jpg")
    cwd = tmp_path / "a" / "b" / "c" / "d"
    cwd.mkdir(parents=True)
    out = subprocess.run([BIN], cwd=cwd, capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    bmp = (tmp_path / "data" / "out.bmp").read_bytes()
    assert len(bmp) == 786486
    want = port.bmp24_bytes(port.decode(open(LENNA, "rb").read())["rgb"])
    assert bmp == want
    # SURVEY.md section 4: BMP the reference itself writes for Lenna
    assert hashlib.sha256(bmp).hexdigest() == "af6996f7f0cb092f8282bd661f95869d6c2c983b364d8722f6ff581eaf5d12e0"
