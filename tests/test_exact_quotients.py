"""The render kernel's division-free quotients (device_path.cuh: div_zero_dividend, div_pi, fmod_pos) against IEEE
division and fmod, over EVERY float32 dividend.  A C++ restatement of the device code (same IEEE operations: products,
fmaf, truncf, selects; compiled with -ffp-contract=off so nothing is fused that the device does not fuse) runs each
check over all 2^32 bit patterns; the reciprocal constants are read from device_path.cuh itself."""
import os
import re
import shutil
import subprocess

import pytest

from conftest import ROOT

SRC = r"""
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <initializer_list>
static inline float bf(uint32_t u) { float f; std::memcpy(&f, &u, 4); return f; }
static inline uint32_t fb(float f) { uint32_t u; std::memcpy(&u, &f, 4); return u; }
static inline bool same(float a, float b) { return fb(a) == fb(b) || (std::isnan(a) && std::isnan(b)); }
static const float kPI = 3.14159265358979323846264338327950288f;

// device_path.cuh, restated
static float div_zero_dividend(float a, float s) {
  const bool z = a == 0.0f && std::fabs(s) > 0.0f;
  const float q = (z ? s : a) / s;
  return z ? bf((fb(a) ^ fb(s)) & 0x80000000u) : q;
}
static float kPI_RCP;
static bool div_pi_window(float a) { const unsigned e = (fb(a) >> 23) & 0xffu; return e - 32u <= 254u - 32u; }
static float div_pi(float a) {
  if (div_pi_window(a)) {
    const float q0 = a * kPI_RCP;
    const float r = std::fmaf(-kPI, q0, a);
    return std::fmaf(r, kPI_RCP, q0);
  }
  return a == 0.0f ? a : a / kPI;
}
static float fmod_pos(float x, float m, float m_rcp) {
  if (!(x < m * 8388608.0f)) return std::fmod(x, m);
  const float q0 = std::trunc(x * m_rcp);
  const float r0 = std::fmaf(-q0, m, x);
  const float q = r0 < 0.0f ? q0 - 1.0f : (r0 >= m ? q0 + 1.0f : q0);
  return std::fmaf(-q, m, x);
}

// every 2^32 pattern, in 2^16 chunks of 2^16 (OpenMP if the compiler has it); returns the number of mismatches and
// prints the first few
template <class F> static unsigned long long all_floats(const char* what, F bad) {
  unsigned long long n_bad = 0;
#pragma omp parallel for schedule(dynamic, 16) reduction(+ : n_bad)
  for (long long hi = 0; hi < 65536; hi++)
    for (uint32_t lo = 0; lo < 65536; lo++) {
      const uint32_t u = (uint32_t)(hi << 16) | lo;
      if (bad(u)) {
        n_bad++;
        if (n_bad <= 3) std::printf("%s: mismatch at 0x%08x\n", what, u);
      }
    }
  return n_bad;
}

int main(int argc, char** argv) {
  const char* mode = argv[1];
  unsigned long long n_bad = 0;
  if (!std::strcmp(mode, "pi")) {
    kPI_RCP = std::strtof(argv[2], nullptr);
    if (kPI_RCP != 1.0f / kPI) { std::printf("kPI_RCP is not RN(1 / kPI)\n"); return 1; }
    unsigned long long fast = 0;
    n_bad = all_floats("x / kPI", [&](uint32_t u) { const float a = bf(u); return !same(div_pi(a), a / kPI); });
    for (uint32_t e = 0; e < 256; e++) fast += div_pi_window(bf(e << 23)) ? (2ull << 23) : 0ull;
    std::printf("dividends on the three-op path: %llu of 2^32\n", fast);
    // the window holds no zero, subnormal, inf or NaN dividend: those take the real division
    for (float a : {0.0f, -0.0f, bf(1u), bf(0x007fffffu), INFINITY, -INFINITY, NAN})
      if (div_pi_window(a)) { std::printf("window admits a special dividend\n"); return 1; }
  } else if (!std::strcmp(mode, "fmod")) {
    const float m = std::strtof(argv[2], nullptr), m_rcp = std::strtof(argv[3], nullptr);
    if (m_rcp != 1.0f / m) { std::printf("reciprocal of %g is not RN(1 / m)\n", m); return 1; }
    n_bad = all_floats("fmod_pos", [&](uint32_t u) {
      const float x = bf(u);
      if ((u >> 31) || !(x < m * 8388608.0f)) return false;    // fmod_pos is called on fabsf(base); beyond, the library fmodf
      return fb(fmod_pos(x, m, m_rcp)) != fb(std::fmod(x, m));
    });
  } else if (!std::strcmp(mode, "zero")) {
    const float sp[] = {0.0f, -0.0f, 1.0f, -1.0f, 1.3f, -0.7f, bf(1u), bf(0x80000001u), bf(0x007fffffu), bf(0x00800000u),
                        bf(0x7f7fffffu), bf(0xff7fffffu), INFINITY, -INFINITY, NAN, -NAN, 3.14159265f, 1e-30f, 1e30f};
    for (float a : sp)
      for (float s : sp)
        if (!same(div_zero_dividend(a, s), a / s)) { n_bad++; std::printf("%a / %a\n", a, s); }
    // a zero dividend over every divisor, and every dividend over a few divisors
    n_bad += all_floats("+-0 / s", [&](uint32_t u) {
      const float s = bf(u);
      return !same(div_zero_dividend(0.0f, s), 0.0f / s) || !same(div_zero_dividend(-0.0f, s), -0.0f / s);
    });
    n_bad += all_floats("a / s", [&](uint32_t u) {
      const float a = bf(u);
      for (float s : {1.3f, -0.7f, bf(1u), INFINITY, 0.0f, NAN})
        if (!same(div_zero_dividend(a, s), a / s)) return true;
      return false;
    });
  }
  std::printf("%s: %llu mismatches\n", mode, n_bad);
  return n_bad ? 1 : 0;
}
"""


def _device_source():
    with open(os.path.join(ROOT, "lumillyrender_b200", "csrc", "device_path.cuh")) as f:
        return f.read()


@pytest.fixture(scope="module")
def checker(tmp_path_factory):
    gxx = shutil.which("g++")
    if not gxx:
        pytest.skip("g++ not available")
    d = tmp_path_factory.mktemp("exact_quotients")
    src, exe = str(d / "check.cpp"), str(d / "check")
    with open(src, "w") as f:
        f.write(SRC)
    base = [gxx, "-std=c++17", "-O2", "-ffp-contract=off", "-fno-fast-math", src, "-o", exe]
    if subprocess.run(base[:1] + ["-fopenmp"] + base[1:], capture_output=True).returncode != 0:
        subprocess.run(base, check=True)
    return exe


def _run(exe, *args):
    out = subprocess.run([exe] + [str(a) for a in args], capture_output=True, text=True, timeout=3600)
    assert out.returncode == 0, out.stdout + out.stderr
    return out.stdout


def _hex_float(name):
    m = re.search(r"\b%s\s*=\s*(0x[0-9a-fA-F.]+p[-+]?\d+)f" % name, _device_source())
    assert m, name
    return float.fromhex(m.group(1))


def test_div_pi_equals_ieee_division_for_every_dividend(checker):
    src = _device_source()
    assert "e - 32u <= 254u - 32u" in src, "the exponent window of div_pi changed: update the restatement"
    out = _run(checker, "pi", repr(_hex_float("kPI_RCP")))
    assert "dividends on the three-op path: %d of 2^32" % ((254 - 32 + 1) * 2 * 2 ** 23) in out, out


@pytest.mark.parametrize("m,name", [(150.0, "li_rcp"), (30.0, "si_rcp"), (300.0, "ci_rcp")])
def test_fmod_pos_equals_fmod_for_every_dividend(checker, m, name):
    _run(checker, "fmod", repr(m), repr(_hex_float(name)))


def test_zero_dividend_quotient_equals_ieee_division(checker):
    _run(checker, "zero")
