"""Prior programs on the host (include/swarm_b200.h group 6): compiling a robot_policy needs NVRTC, not a GPU.  The image is an
sm_100a CUBIN with the three entry points, compiled without FMA contraction; compile errors come back with NVRTC's log; the
library does not link NVRTC or libcuda."""
import ctypes as C
import os
import re
import shutil
import subprocess

import pytest

from marl_llm_b200 import _lib
from marl_llm_b200 import prior_program as pp
from marl_llm_b200.build import build_library

NVRTC = pp.find_nvrtc()
pytestmark = pytest.mark.skipif(NVRTC is None, reason="NVRTC (libnvrtc.so.12) not installed")
CUOBJDUMP = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"

PROBE = """#include "swarm_prior_api.cuh"
__device__ void robot_policy(const swarm_agent &a, double out[2]) {
    out[0] = a.x * a.x + a.y * a.y;
    out[1] = 0.0;
}
"""
SYNTAX_ERROR = """#include "swarm_prior_api.cuh"
__device__ void robot_policy(const swarm_agent &a, double out[2]) {
    out[0] = a.x
    out[1] = a.y;
}
"""
NO_POLICY = """#include "swarm_prior_api.cuh"
__device__ void robot_policy_v2(const swarm_agent &a, double out[2]) { out[0] = a.x; out[1] = a.y; }
"""


@pytest.fixture(scope="module")
def lib():
    build_library()
    return _lib.load()


@pytest.fixture(scope="module")
def shipped(lib):
    return pp.compile_source(pp.reference_prior_source(), NVRTC)


def raw_compile(lib, source, path=NVRTC, image_cap=0, with_image=False):
    size, log = C.c_int64(-1), C.create_string_buffer(1 << 16)
    img = C.create_string_buffer(max(image_cap, 1)) if with_image else None
    rc = lib.swarm_prior_compile(source.encode(), path.encode() if path else None, img, image_cap, C.byref(size), log, 1 << 16)
    return rc, size.value, log.value.decode(), img


def sass(image, tmp_path, name):
    f = tmp_path / name
    f.write_bytes(image)
    if not os.path.isfile(CUOBJDUMP):
        pytest.skip("cuobjdump not installed")
    return subprocess.run([CUOBJDUMP, "-sass", str(f)], check=True, capture_output=True, text=True).stdout


def test_the_shipped_program_compiles_to_an_sm100a_cubin_with_three_entry_points(shipped, tmp_path):
    image, log = shipped
    assert image[:4] == b"\x7fELF" and image[4] == 2          # 64-bit ELF, not PTX text
    assert b".version" not in image[:64]
    text = sass(image, tmp_path, "reference_prior.cubin")
    assert "code for sm_100a" in text, text[:400]
    funcs = set(re.findall(r"Function : (\w+)", text))
    assert funcs == {"swarm_prior_f32", "swarm_prior_f64", "swarm_prior_actions"}, funcs


def test_products_are_not_contracted_into_fmas(lib, tmp_path):
    rc, size, log, _ = raw_compile(lib, PROBE)
    assert rc == _lib.SWARM_OK, log
    rc, size2, _, img = raw_compile(lib, PROBE, image_cap=size, with_image=True)
    assert rc == _lib.SWARM_OK and size2 == size
    text = sass(img.raw[:size], tmp_path, "probe.cubin")
    for fn in re.split(r"Function : ", text)[1:]:
        ops = re.findall(r"\b(DMUL|DADD|DFMA)\b", fn)
        # x*x + y*y (and the wrapper's dx*dx + dy*dy) as two products and a sum: the probe has no division or sqrt, so no DFMA
        assert "DFMA" not in ops and ops.count("DMUL") >= 2 and "DADD" in ops, ops


def test_image_size_query_and_short_buffer(lib, shipped):
    rc, size, _, _ = raw_compile(lib, pp.reference_prior_source())
    assert rc == _lib.SWARM_OK and size == len(shipped[0])
    rc, _, _, _ = raw_compile(lib, pp.reference_prior_source(), image_cap=size - 1, with_image=True)
    assert rc == _lib.SWARM_ERR_INVALID and b"image_cap" in lib.swarm_last_error()


def test_a_syntax_error_is_reported_with_its_line(lib):
    rc, _, log, _ = raw_compile(lib, SYNTAX_ERROR)
    assert rc == _lib.SWARM_ERR_INVALID
    assert "robot_policy.cu(4): error" in log, log
    with pytest.raises(_lib.SwarmError, match=r"robot_policy\.cu\(4\): error"):
        pp.PriorProgram(SYNTAX_ERROR)


def test_a_missing_robot_policy_is_reported(lib):
    rc, _, log, _ = raw_compile(lib, NO_POLICY)
    assert rc == _lib.SWARM_ERR_INVALID
    assert re.search(r"\(\d+\): error: identifier \"robot_policy\" is undefined", log), log
    with pytest.raises(_lib.SwarmError, match="robot_policy"):
        pp.PriorProgram(NO_POLICY)


def test_a_missing_nvrtc_is_unsupported_and_names_the_path(lib):
    rc, _, _, _ = raw_compile(lib, PROBE, path="/nonexistent/dir/libnvrtc.so.12")
    assert rc == _lib.SWARM_ERR_UNSUPPORTED
    assert b"/nonexistent/dir/libnvrtc.so.12" in lib.swarm_last_error()


def test_null_arguments_are_invalid(lib):
    size = C.c_int64()
    assert lib.swarm_prior_compile(None, None, None, 0, C.byref(size), None, 0) == _lib.SWARM_ERR_INVALID
    assert lib.swarm_prior_compile(PROBE.encode(), NVRTC.encode(), None, 0, None, None, 0) == _lib.SWARM_ERR_INVALID
    h = C.c_void_p()
    assert lib.swarm_prior_program_create(0, None, 0, C.byref(h)) == _lib.SWARM_ERR_INVALID
    junk = b"not a cubin" * 10
    assert lib.swarm_prior_program_create(0, junk, len(junk), C.byref(h)) == _lib.SWARM_ERR_INVALID
    assert lib.swarm_set_prior_program(None, None) == _lib.SWARM_ERR_INVALID
    assert lib.swarm_prior_program_actions(None, None, None, None) == _lib.SWARM_ERR_INVALID


def test_the_library_links_neither_nvrtc_nor_libcuda(lib):
    readelf = shutil.which("readelf")
    if readelf is None:
        pytest.skip("readelf not installed")
    out = subprocess.run([readelf, "-d", _lib.LIB_PATH], check=True, capture_output=True, text=True).stdout
    needed = re.findall(r"\(NEEDED\).*\[(.+)\]", out)
    assert needed and not [n for n in needed if "nvrtc" in n or n.startswith("libcuda.")], needed
