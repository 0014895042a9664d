"""CPU: the C-ABI library loads here (no GPU) and exports every symbol that
include/rcc_ba.h declares; compute entry points fail loudly without a device."""
import ctypes
import os
import re

from robot_camera_calibration_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    src = open(os.path.join(ROOT, "include", "rcc_ba.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(rcc_[a-z0-9_]+)\s*\(", src)))


def test_header_symbols_are_exported_and_bound():
    names = _declared()
    assert len(names) >= 35
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/rcc_ba.h but not exported"
    assert set(names) == set(_lib.SIGNATURES), set(names) ^ set(_lib.SIGNATURES)


def test_library_identifies_itself():
    lib = _lib.load()
    v = lib.rcc_ba_version().decode()
    assert "sm_100a" in v and "fp64" in v


def test_bad_arguments_are_rejected_without_a_device():
    lib = _lib.load()
    h = ctypes.c_void_p()
    assert lib.rcc_ba_create(None, ctypes.byref(h)) == _lib.RCC_BAD_ARG
    opt = _lib.Options(model=0, n_views=0, n_markers=3, n_cameras=1, n_obs_blocks=0, device=0, eliminate=0)
    assert lib.rcc_ba_create(ctypes.byref(opt), ctypes.byref(h)) == _lib.RCC_BAD_ARG
    assert lib.rcc_ba_linearize(None, None) == _lib.RCC_BAD_ARG


def test_no_cpu_fallback():
    """Without a CUDA device creating a problem must fail loudly (RCC_CUDA_ERROR),
    never fall back to a CPU path.  Checked in a child process that sees no device,
    so that it holds on a GPU machine as well."""
    import subprocess
    import sys
    child = ("from robot_camera_calibration_b200 import _lib\n"
             "from robot_camera_calibration_b200.problem import BAProblem\n"
             "try:\n"
             "    BAProblem(4, 4, 1, 0)\n"
             "except _lib.RccError as e:\n"
             "    assert e.status == _lib.RCC_CUDA_ERROR, e\n"
             "    assert 'no CPU fallback' in str(e), e\n"
             "else:\n"
             "    raise SystemExit('a problem was created without a device')\n")
    r = subprocess.run([sys.executable, "-c", child], cwd=ROOT, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "robot_camera_calibration_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".cpp")):
                txt = open(os.path.join(dirpath, f)).read()
                assert "ba_oracle" not in txt and "cpu_baseline" not in txt and "cpu_restatement" not in txt, f


def test_header_is_plain_c_and_a_c_caller_links(tmp_path):
    """include/rcc_ba.h is the drop-in boundary: it must compile as C99 (no C++, no torch types) and a C
    translation unit written like INTEGRATION.md's stub must link against librcc_ba.so."""
    import subprocess
    from robot_camera_calibration_b200 import _lib as L
    src = tmp_path / "caller.c"
    src.write_text(
        '#include "rcc_ba.h"\n'
        "int main(void) {\n"
        "  rcc_ba_options opt = {RCC_MODEL_SINGLE, 2, 2, 1, 0, 0, RCC_ELIM_AUTO};\n"
        "  rcc_ba_problem* p = 0;\n"
        "  rcc_lm_options lm; rcc_lm_default_options(&lm);\n"
        "  /* no device on the build box: creation must fail cleanly, never fall back */\n"
        "  int rc = rcc_ba_create(&opt, &p);\n"
        "  return (rc == RCC_OK) ? (rcc_ba_destroy(p), 0) : (rcc_ba_last_error(0) ? 0 : 1);\n"
        "}\n")
    exe = tmp_path / "caller"
    inc = os.path.join(ROOT, "include")
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-pedantic", "-I", inc, str(src), "-o", str(exe),
                    L.LIB_PATH, "-Wl,-rpath," + os.path.dirname(L.LIB_PATH), "-Wl,-rpath,/usr/local/cuda/lib64"],
                   check=True)
    assert subprocess.run([str(exe)]).returncode == 0
