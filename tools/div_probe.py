"""Cost of one IEEE fp32 division by operand class on the GPU: which classes leave the inline sequence for the slow path.

  python tools/div_probe.py            (needs nvcc and a CUDA device; builds into a temporary directory)

Compiled with the render kernel's flags (-prec-div=true -fmad=false), so every `a / b` is MUFU.RCP + FFMA + FCHK with
a call to __cuda_sm3x_div_rn_noftz_f32_slowpath when FCHK fires.  One warp runs a dependent chain of N quotients per
class, all lanes with the same operands, and times it with clock64(); the dividend of each step depends on the previous
quotient through a mask that is zero at run time, so the operands stay those of the class.  The class "no division"
(a * b in the same chain) is the loop's own cost; the table gives cycles per step with and without it."""
import ctypes as C
import os
import shutil
import subprocess
import sys
import tempfile

SRC = r"""
#include <cstdint>
__global__ void chain(const float* a, const float* b, int n_classes, int iters, unsigned mask, long long* cycles, float* sink) {
  for (int k = 0; k < n_classes; k++) {
    float x = a[k];
    const float y = b[k];
    const unsigned ax = __float_as_uint(x);
    float acc = 0.0f;
    __syncwarp();
    const long long t0 = clock64();
#pragma unroll 4
    for (int i = 0; i < iters; i++) {
      const float q = (k == 0) ? x * y : x / y;
      acc = q;
      x = __uint_as_float(ax ^ (__float_as_uint(q) & mask));
    }
    __syncwarp();
    const long long t1 = clock64();
    if (threadIdx.x == 0) { cycles[k] = t1 - t0; sink[k] = acc; }
  }
}
extern "C" int probe(const float* a, const float* b, int n, int iters, long long* cycles, float* quot) {
  float *da, *db, *ds; long long* dc;
  cudaMalloc(&da, n * 4); cudaMalloc(&db, n * 4); cudaMalloc(&ds, n * 4); cudaMalloc(&dc, n * 8);
  cudaMemcpy(da, a, n * 4, cudaMemcpyHostToDevice);
  cudaMemcpy(db, b, n * 4, cudaMemcpyHostToDevice);
  for (int rep = 0; rep < 2; rep++) chain<<<1, 32>>>(da, db, n, iters, 0u, dc, ds);   // the first launch warms up
  int e = (int)cudaDeviceSynchronize();
  cudaMemcpy(cycles, dc, n * 8, cudaMemcpyDeviceToHost);
  cudaMemcpy(quot, ds, n * 4, cudaMemcpyDeviceToHost);
  cudaFree(da); cudaFree(db); cudaFree(ds); cudaFree(dc);
  return e;
}
"""

PI = 3.14159265358979323846
# (name, dividend, divisor); the first row is the loop without a division
CLASSES = [
    ("no division (a * b)", 1.5, 0.7),
    ("normal / normal", 1.5, 0.7),
    ("normal / norm-like", 0.6, 1.3),
    ("+0 / normal", 0.0, 1.3),
    ("-0 / normal", -0.0, 1.3),
    ("3 pi / pi", 3.0 * PI, PI),
    ("x / pi (x = 0.25)", 0.25, PI),
    ("huge / normal (3e38 / 1.5)", 3.0e38, 1.5),
    ("tiny / normal (1e-37 / 0.7)", 1.0e-37, 0.7),
    ("denormal / normal (1e-40 / 0.7)", 1.0e-40, 0.7),
    ("x / 150 (x = 1234.5)", 1234.5, 150.0),
]


def main():
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    iters = 4096
    with tempfile.TemporaryDirectory() as tmp:
        cu, so = os.path.join(tmp, "div_probe.cu"), os.path.join(tmp, "div_probe.so")
        with open(cu, "w") as f:
            f.write(SRC)
        subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-fmad=false", "-prec-div=true", "-shared",
                        "-Xcompiler", "-fPIC", "-o", so, cu], check=True)
        lib = C.CDLL(so)
        n = len(CLASSES)
        a = (C.c_float * n)(*[c[1] for c in CLASSES])
        b = (C.c_float * n)(*[c[2] for c in CLASSES])
        cyc = (C.c_longlong * n)()
        quot = (C.c_float * n)()
        rc = lib.probe(a, b, n, iters, cyc, quot)
        if rc != 0:
            sys.exit("div_probe: CUDA error %d" % rc)
    base = cyc[0] / iters
    print("%-34s %12s %14s  %s" % ("class", "cycles/step", "minus loop", "last quotient"))
    for k, (name, _, _) in enumerate(CLASSES):
        per = cyc[k] / iters
        print("%-34s %12.1f %14.1f  %r" % (name, per, per - base if k else 0.0, quot[k]))


if __name__ == "__main__":
    main()
