"""kernel_ready (csrc/common.cuh), the one place that opts a kernel in to more than 48 KB of dynamic shared memory on a
device: a request the device cannot grant is refused with status -3 and a message that names the kernel, and a granted
one lets the kernel launch with that much.  A small host program includes the header and links libader_b200.so; it
needs a CUDA device to run and is skipped without one."""
import os
import subprocess

import pytest

from ader_b200 import build

PROGRAM = r"""
#include "common.cuh"
__global__ void k_too_big() {}
__global__ void k_fits(float* out) { extern __shared__ float s[]; s[threadIdx.x] = 1.f; __syncthreads(); out[0] = s[0]; }
int main() {
  const int refused = ader::kernel_ready<k_too_big>(1 << 30, "k_too_big");
  printf("refused %d %s\n", refused, ader_last_error());
  const int granted = ader::kernel_ready<k_fits>(100 * 1024, "k_fits");
  const int again = ader::kernel_ready<k_fits>(100 * 1024, "k_fits");
  float* out = nullptr;
  cudaMalloc(&out, sizeof(float));
  k_fits<<<1, 32, 100 * 1024>>>(out);
  const cudaError_t e = cudaDeviceSynchronize();
  printf("granted %d %d %s\n", granted, again, cudaGetErrorName(e));
  cudaFree(out);
  return 0;
}
"""


def test_refused_opt_in_names_the_kernel(tmp_path):
    torch = pytest.importorskip("torch")
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    lib = build.build()
    src, exe = tmp_path / "probe.cu", tmp_path / "probe"
    src.write_text(PROGRAM)
    lib_dir = os.path.dirname(lib)
    subprocess.run([build._nvcc(), "-gencode", "arch=compute_100a,code=sm_100a", "-std=c++17", "-I", build.CSRC, str(src), "-o", str(exe),
                    "-L", lib_dir, "-lader_b200", "-Xlinker", "-rpath=" + lib_dir], check=True)
    lines = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.splitlines()
    refused, granted = lines[0].split(" ", 2), lines[1].split()
    assert refused[1] == "-3"
    assert refused[2].startswith("k_too_big: cannot reserve 1073741824 B of shared memory on device 0: ")
    assert granted[1:] == ["0", "0", "cudaSuccess"]
