"""mlx5 wire format against an independent source: DOCA GPUNetIO's own definitions, as shipped in the NCCL wheel
(nvidia-nccl-cu12 2.28.9, BSD-3-Clause; a verbatim copy is kept in tests/golden so the check never depends on what
is installed).  See tests/native/wire_crosscheck.cc (every assertion is a static_assert: compiling IS the test)."""
import shutil
import subprocess
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent


def _doca_header():
    return Path(__file__).resolve().parent / "golden" / "doca_gpunetio_verbs_def.h"


@pytest.mark.skipif(shutil.which("g++") is None, reason="no host compiler")
def test_layouts_opcodes_and_flags_agree_with_doca_gpunetio():
    hdr = _doca_header()
    cmd = ["g++", "-std=c++17", "-fsyntax-only", "-fpermissive", "-w", f"-I{ROOT / 'rocnrdma_b200' / 'csrc'}",
           f'-DDOCA_VERBS_DEF_H="{hdr}"', str(ROOT / "tests" / "native" / "wire_crosscheck.cc")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stderr[-3000:]


def test_the_crosscheck_can_fail(tmp_path):
    """Negative control: shift one of our fields and the same translation unit must stop compiling."""
    hdr = _doca_header()
    if shutil.which("g++") is None:
        pytest.skip("no host compiler")
    src = (ROOT / "rocnrdma_b200" / "csrc" / "wire" / "mlx5_wire.h").read_text()
    broken = src.replace("  uint8_t signature;\n  uint8_t rsvd[2];\n  uint8_t fm_ce_se;", "  uint8_t signature;\n  uint8_t fm_ce_se;\n  uint8_t rsvd[2];", 1)
    assert broken != src
    (tmp_path / "wire").mkdir()
    (tmp_path / "wire" / "mlx5_wire.h").write_text(broken)
    cmd = ["g++", "-std=c++17", "-fsyntax-only", "-fpermissive", "-w", f"-I{tmp_path}", f'-DDOCA_VERBS_DEF_H="{hdr}"',
           str(ROOT / "tests" / "native" / "wire_crosscheck.cc")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=120)
    assert r.returncode != 0 and "fm_ce_se" in r.stderr
