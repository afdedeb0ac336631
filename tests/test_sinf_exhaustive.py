"""The device sine and cosine against libm for EVERY float.

knaster's SinNumeric is `f32::sin` and PolyBlep's Cosine `f32::cos`, i.e. the platform libm's sinf / cosf (osc.rs:264,
polyblep.rs:247); csrc/sinf_glibc.h restates glibc's algorithms (sinf in three forms: the general one for every float, the
|y| < 120 one and the leaner one the FM kernels run; cosf in one).  A float has only 2^32 values: tools/sinf_exhaustive.cpp runs
them (host instantiation, the same f64 and integer operations the device executes) over all bit patterns -- the |y| < 120 forms
over their domain -- and counts the results that differ from libm's by even one bit (NaN counts as equal to NaN).
"""
import json
import os
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_sine_and_cosine_restatements_equal_libm_for_every_float(tmp_path):
    exe = tmp_path / "sinf_exhaustive"
    fma = "fma" in open("/proc/cpuinfo").read().split("flags", 1)[-1].split("\n", 1)[0].split()
    cmd = ["g++", "-O2", "-ffp-contract=off", "-pthread", "-I" + os.path.join(ROOT, "knaster_b200", "csrc"),
           os.path.join(ROOT, "tools", "sinf_exhaustive.cpp"), "-o", str(exe)] + (["-mfma"] if fma else [])
    subprocess.run(cmd, check=True)
    # without hardware FMA the software fma() is ~50x slower: a stride keeps the run bounded there
    stride = 1 if fma else 64
    out = subprocess.run([str(exe), str(stride)], check=True, capture_output=True, text=True, timeout=900).stdout
    r = json.loads(out)
    print(out.strip())
    assert r["arguments"] >= (1 << 32) // stride
    assert r["inrange_arguments"] >= 2 * 0x42F00000 // stride
    if r["fma_cpu"]:
        # glibc's ifunc runs __sinf_fma / __cosf_fma here: the restatements' fused operations are the same ones
        assert r["sin_mismatches"] == 0 and r["cos_mismatches"] == 0, r
        assert r["inrange_mismatches"] == 0 and r["lean_mismatches"] == 0, r
    else:
        # an un-fused libm differs from the fused one in about a dozen of the 2.2e9 results below 120
        assert r["inrange_mismatches"] <= 32 and r["lean_mismatches"] <= 32, r
        assert r["sin_mismatches"] <= 64 and r["cos_mismatches"] <= 64, r
    assert r["lean_zero_sign_only"] <= 1, r  # sin(-0.0): +0.0 in the lean form
