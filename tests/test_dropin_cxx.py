"""The C++ drop-in: the reference's README example compiled against include/signal_packer.h and
linked with librspt_packer.so (which reaches CUDA only through the C ABI)."""
import os
import re
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _build_example(tmp_path):
    from rspt_b200.build import build
    build()
    exe = str(tmp_path / "dropin_example")
    lib = os.path.join(ROOT, "rspt_b200")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-I", os.path.join(ROOT, "include"), "-o", exe,
                           os.path.join(ROOT, "tests", "cxx", "dropin_example.cpp"), "-L", lib,
                           "-lrspt_packer", "-lrspt_gpu", f"-Wl,-rpath,{lib}"])
    return exe


def test_dropin_links_and_refuses_without_gpu(tmp_path):
    """The example builds against the drop-in header; without a CUDA device (none visible to the
    process) the factory reports the failure and returns null (exit code 2) -- there is no CPU fallback."""
    exe = _build_example(tmp_path)
    r = subprocess.run([exe], capture_output=True, text=True, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert r.returncode == 2 and "rspt_gpu_create failed (-5)" in r.stdout


@pytest.mark.gpu
def test_dropin_readme_example_on_gpu(tmp_path):
    exe = _build_example(tmp_path)
    r = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    m = re.search(r"compressed_size: (\d+) consumed: (\d+) rc: 0 roundtrip: ok", r.stdout)
    assert m and m.group(1) == m.group(2) == "2028", r.stdout      # BASELINE.md section 3
    m = re.search(r"hadamard: (\d+) dct: (\d+) hzr: (\d+)", r.stdout)
    assert m and (m.group(1), m.group(2), m.group(3)) == ("1013", "114", "12010"), r.stdout
