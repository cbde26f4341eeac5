"""Host side of the multi-view render, without a GPU: the C++ frame program builds against the host API, and the
Python binding mirrors the C-ABI's new entry point and the rt_stats field it reports."""
import ctypes as C
import os
import subprocess


def test_views_program_compiles_against_the_host_api(rtb, built, tmp_path):
    host = os.path.join(rtb.REPO_ROOT, "raytracing-practice_b200", "host")
    libdir = os.path.dirname(rtb.CUDA_LIB_PATH)
    exe = str(tmp_path / "views")
    r = subprocess.run(["g++", "-std=c++11", "-O1", "-Wall", "-Werror", "-I", host, "-I", os.path.join(rtb.REPO_ROOT, "include"),
                        os.path.join(rtb.REPO_ROOT, "tests", "cpp", "views_main.cpp"), "-L", libdir, "-lrt_b200", "-Wl,-rpath," + libdir, "-o", exe],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    r = subprocess.run([exe], capture_output=True, text=True)
    assert r.returncode == 2 and "usage" in r.stderr


def test_render_views_binding(rtb, built):
    lib = rtb.cuda_lib()
    assert hasattr(lib, "rt_render_views") and "rt_render_views" in rtb.C_ABI_SYMBOLS
    # rt_stats.reserved0 became n_views: same size, same offset
    assert rtb.rt_stats.n_views.offset == rtb.rt_stats.n_boxes.offset + 4
    assert C.sizeof(rtb.rt_stats) == lib.rt_abi_sizeof(9)
    # a null context is refused before anything else
    assert lib.rt_render_views(None, 1, None, None) == rtb.RT_ERR_INVALID
