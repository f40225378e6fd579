"""The C ABI driven from plain C99 (tests/c_abi/abi_smoke.c): the header is valid C, the shared library links with a C
compiler, and the error / no-device behaviour is a status code plus a message — what a JNA, Panama or cgo binding
relies on.  With no device visible the program must report RT_ERR_NODEVICE (exit 3); on a GPU it renders."""
import os
import shutil
import subprocess

import pytest

from raytrace_clj_b200 import build as rtbuild

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "c_abi", "abi_smoke.c")


def _build(tmp_path):
    lib = rtbuild.build_library()
    exe = str(tmp_path / "abi_smoke")
    cc = shutil.which("gcc") or shutil.which("cc")
    assert cc, "no C compiler"
    libdir = os.path.dirname(lib)
    subprocess.check_call([cc, "-std=c11", "-Wall", "-Wextra", "-Werror", "-pedantic", "-I", os.path.join(ROOT, "include"), SRC,
                           "-o", exe, "-L", libdir, "-lraytrace_b200", "-lm", f"-Wl,-rpath,{libdir}"])
    return exe


def test_header_is_plain_c_and_library_links_from_c(tmp_path):
    exe = _build(tmp_path)
    # the program sees no device (CUDA_VISIBLE_DEVICES empty), so a machine with GPUs checks the refusal too
    res = subprocess.run([exe], capture_output=True, text=True, timeout=120, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert res.returncode == 3, (res.returncode, res.stdout, res.stderr)
    assert "nodevice" in res.stdout and "no CPU fallback" in res.stdout


@pytest.mark.gpu
def test_c_program_renders_through_the_abi(tmp_path):
    exe = _build(tmp_path)
    res = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert res.returncode == 0, (res.returncode, res.stdout, res.stderr)
    assert res.stdout.startswith("ok:")
