"""The device arithmetic under the engine's bit-identical results, on the GPU, over whole domains (tools/devmath_exhaustive.cu).

A float has 2^32 values; the harness runs the device helpers (compiled from the kernels' own headers with the library's numeric
flags) over all of them, or over every value of their domain, and compares with libm or IEEE arithmetic:
  a/b  kn_sinf and kn_cosf against glibc sinf / cosf for every float; the |y| < 120 sine forms (inrange, lean, lean_n<32>)
       against kn_sinf for every |y| < 120;
  c    div_rc(n, d, div_prep(d)) against IEEE n / d for every pair of significands n, d in [1, 2).  While q0, the FMA remainder
       and the correction stay normal their rounding depends on the significands only, so these 2^46 pairs cover every normal
       quotient the saw (blep window) and FM (v / sr) paths form.  And render_fm2's increment expression for every finite v at
       seven sample rates;
  d    saw_fast_tick against polyblep_saw_tick and saw_eval2 against saw_eval, every t in [0, 1) at 64 increments;
  e    wrap_threshold for every dt in [2^-20, 1/4), and wrap_flag around it;
  f    kn_tanf / kn_expf / kn_powf: at most 1 ulp from glibc, correctly rounded except where undecidable, fractions printed.
"""
import json
import os
import shutil
import subprocess

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NVCC = os.environ.get("NVCC", shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc")
# the library's numeric flags (knaster_b200/csrc/Makefile)
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-fmad=false", "-prec-div=true", "-prec-sqrt=true",
         "-ftz=false"]


@pytest.fixture(scope="module")
def result(tmp_path_factory):
    exe = tmp_path_factory.mktemp("devmath") / "devmath_exhaustive"
    subprocess.run([NVCC, *FLAGS, "-I" + os.path.join(ROOT, "knaster_b200", "csrc"), os.path.join(ROOT, "tools", "devmath_exhaustive.cu"),
                    "-o", str(exe), "-lpthread"], check=True)
    out = subprocess.run([str(exe)], check=True, capture_output=True, text=True, timeout=900).stdout
    print(out.strip())
    return json.loads(out.strip().splitlines()[-1])


def test_sine_and_cosine_equal_glibc_for_every_float(result):
    for fn in ("sin", "cos"):
        assert result[fn]["arguments"] == 1 << 32, result[fn]
        assert result[fn]["mismatches"] == 0, (fn, result[fn])
    assert result["sin_inrange"]["mismatches"] == 0, result["sin_inrange"]
    for form in ("sin_lean", "sin_lean_n"):
        assert result[form]["mismatches"] == 0, (form, result[form])
        assert result[form]["aux"] <= 1, (form, result[form])   # sin(-0.0) = +0.0 in the lean forms


def test_hoisted_division_is_correctly_rounded(result):
    assert result["div_pairs"]["mismatches"] == 0, result["div_pairs"]
    # render_fm2's increment: exact for every normal quotient; where v / sr is subnormal (|v| < 6e-34) the scaled form may
    # round twice, and a 1e-45 increment cannot move a phase
    assert result["div_fm"]["mismatches"] == 0, result["div_fm"]


def test_straight_line_saw_equals_reference_order_saw(result):
    assert result["saw_dts"] == 64
    assert result["saw_tick"]["mismatches"] == 0, result["saw_tick"]
    assert result["saw_pair"]["mismatches"] == 0, result["saw_pair"]


def test_wrap_threshold_for_every_increment(result):
    assert result["wrap_threshold"]["mismatches"] == 0, result["wrap_threshold"]
    assert result["wrap_flag"]["mismatches"] == 0, result["wrap_flag"]


@pytest.mark.parametrize("fn", ["tan", "exp", "pow_db", "pow_sample"])
def test_filter_coefficient_functions_within_one_ulp_of_glibc(result, fn):
    r = result[fn]
    print(fn, {k: r[k] for k in ("arguments", "fraction_differs_from_glibc", "fraction_glibc_not_correctly_rounded", "undecided")})
    assert r["arguments"] >= (1 << 24 if fn == "pow_sample" else 1 << 30), r
    assert r["over_1ulp_from_glibc"] == 0, r
    assert r["not_correctly_rounded"] == 0, r
    assert r["fraction_differs_from_glibc"] < 0.01, r
