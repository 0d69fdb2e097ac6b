"""CPU emulation of the CUDA tile code (threads as loops, phases as barriers): the same source that the
sm_100a kernels compile is run on the host and compared with the oracle. Catches indexing / arithmetic
formulation bugs without a GPU. (Not a product path: built only here.)"""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _build_and_run(tmp_path, src, exe, args=(), defs=()):
    import oracle_lib

    oracle_lib.build_oracle()
    out = str(tmp_path / exe)
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-DGL_FORCE_32BIT_PATH", *defs, "-o", out,
                           os.path.join(ROOT, "tests", "emu", src), "-L" + os.path.join(ROOT, "oracle"),
                           "-lgl_oracle", "-Wl,-rpath," + os.path.join(ROOT, "oracle"), "-pthread"])
    r = subprocess.run([out, *args], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    return r.stdout


def test_field_and_poseidon_device_formulation_on_host(tmp_path):
    assert "EMU OK" in _build_and_run(tmp_path, "field_poseidon_emu.cpp", "gl_fp_emu")


def test_ntt_tiles_forward_inverse_lde_on_host(tmp_path):
    # log_n 1..13: single-pass (<= 12) and two-pass (13) plans; forward, inverse and leaf-major coset LDE
    assert "EMU OK" in _build_and_run(tmp_path, "ntt_emu.cpp", "gl_ntt_emu", ["13"])


def test_poseidon_fp64_pipe_formulation_on_host(tmp_path):
    # the FP64 MDS layers and the FP64-resident partial rounds (device default) with IEEE doubles on the CPU:
    # bit-exact vs both oracle forms (fast and naive partial rounds), limb magnitudes stay below 2^51
    out = _build_and_run(tmp_path, "poseidon_f64_emu.cpp", "gl_f64_emu", ["60000"], defs=["-DGL_FP64_ON_HOST"])
    assert "POSEIDON F64 EMU OK" in out, out
