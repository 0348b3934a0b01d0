"""glibm::pow_half (csrc/glibm.cuh, the device pow(x, 0.5) of the element-set forms of calculate_state_information,
satellite_function.py:309) compiled for the host with g++ and compared bit for bit with the system libm's pow(x, 0.5).
CPU test: no GPU, no oracle involved."""
import ctypes
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "ppo-rl-satellite_b200", "csrc")

SRC = r"""
#include "glibm.cuh"
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstdint>

static double (*volatile libm_pow)(double, double) = pow;

static uint64_t s = 0x9E3779B97F4A7C15ull;
static uint64_t next() { s ^= s << 13; s ^= s >> 7; s ^= s << 17; return s; }

int main(int argc, char** argv) {
    const long n = atol(argv[1]);
    long bad = 0, checked = 0;
    auto check = [&](double x) {
        const double want = libm_pow(x, 0.5), got = glibm::pow_half(x);
        const bool same = (std::isnan(want) && std::isnan(got)) || glibm::bits_(want) == glibm::bits_(got);
        if (!same && bad < 10) printf("mismatch x=%a libm=%a glibm=%a\n", x, want, got);
        bad += !same; ++checked;
    };
    for (long k = 0; k < n; ++k) {
        check(glibm::dbl_(next() & 0x7fffffffffffffffull));                    // every positive bit pattern, incl. subnormal / inf / nan
        check(std::ldexp(1.0 + (double)(next() >> 11) * 0x1p-53, (int)(next() % 80) - 40));   // O(1) magnitudes
        check(1.0 + ((double)(next() >> 11) * 0x1p-53 - 0.5) * 0x1p-40);        // near 1 (|0.5 log x| < 2^-54 exit)
        check(3.986e14 / (6.0e6 + (double)(next() >> 11) * 0x1p-53 * 6.0e7));   // miu / p of the element-set forms
    }
    const double special[] = {0.0, -0.0, INFINITY, -INFINITY, NAN, -1.0, 4.0, 0.25, 1.0, 0x1p-1074, 0x1p-1022, 1.7976931348623157e308};
    for (double x : special) check(x);
    printf("checked %ld mismatches %ld\n", checked, bad);
    return bad != 0;
}
"""


def _glibc_version():
    f = ctypes.CDLL(None).gnu_get_libc_version
    f.restype = ctypes.c_char_p
    return f().decode()


def test_pow_half_bit_identical_to_system_libm(tmp_path):
    if not _glibc_version().startswith("2.39"):
        pytest.skip("glibm.cuh restates glibc 2.39; this host runs %s" % _glibc_version())
    src = tmp_path / "pow_half.cpp"
    src.write_text(SRC)
    exe = str(tmp_path / "pow_half")
    subprocess.run(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fno-builtin-pow", "-mfma", "-I", CSRC, str(src),
                    "-o", exe, "-lm"], check=True)
    r = subprocess.run([exe, "500000"], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout[-2000:]
    assert r.stdout.strip().endswith("mismatches 0") and "checked 2000012" in r.stdout
