// Test helper of tests/test_gpu_param_reset_device.py: the device's fsin_dev / fcos_dev (geometry_device.cuh) against the
// host's (float)std::sin / std::cos((double)x), the functions build_geometry calls (geometry.cpp), on every float of a range
// of bit patterns.  The host half is compiled with the flags geometry.cpp gets (-ffp-contract=off -fno-fast-math -O2).
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstring>
#include <thread>
#include <vector>

#include "../rlfluidcontrol_b200/csrc/geometry_device.cuh"

namespace {

float host_sin(float x) { return (float)std::sin((double)x); }
float host_cos(float x) { return (float)std::cos((double)x); }

__global__ void k_trig(unsigned base, unsigned count, unsigned* out) {
  for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < count; i += gridDim.x * blockDim.x) {
    const float x = __uint_as_float(base + i);
    out[2 * (size_t)i] = __float_as_uint(rlfc::fsin_dev(x));
    out[2 * (size_t)i + 1] = __float_as_uint(rlfc::fcos_dev(x));
  }
}

unsigned bits(float f) { unsigned u; std::memcpy(&u, &f, 4); return u; }

}  // namespace

extern "C" {

// Every float with bit pattern lo .. hi (inclusive, one sign): stats[0] / stats[1] = sin / cos mismatches, stats[2] = floats
// compared; first[0..7] = the first mismatching bit patterns (sin then cos, 4 each, 0xffffffff = none).  Returns 0 or a
// CUDA error code.
int trig_check(unsigned lo, unsigned hi, long long* stats, unsigned* first) {
  const unsigned chunk = 1u << 26;
  unsigned* d = nullptr;
  if (cudaMalloc(&d, (size_t)2 * chunk * sizeof(unsigned)) != cudaSuccess) return 1;
  std::vector<unsigned> h((size_t)2 * chunk);
  std::atomic<long long> ms{0}, mc{0};
  for (int k = 0; k < 8; k++) first[k] = 0xffffffffu;
  std::atomic<int> nfs{0}, nfc{0};
  const int nth = (int)std::max(1u, std::thread::hardware_concurrency());
  int rc = 0;
  for (unsigned long long base = lo; base <= hi; base += chunk) {
    const unsigned count = (unsigned)std::min<unsigned long long>(chunk, (unsigned long long)hi - base + 1);
    k_trig<<<4096, 256>>>((unsigned)base, count, d);
    if (cudaMemcpy(h.data(), d, (size_t)2 * count * sizeof(unsigned), cudaMemcpyDeviceToHost) != cudaSuccess) { rc = 2; break; }
    std::vector<std::thread> th;
    for (int t = 0; t < nth; t++)
      th.emplace_back([&, t] {
        long long s = 0, c = 0;
        for (unsigned i = t; i < count; i += nth) {
          float x;
          const unsigned xb = (unsigned)base + i;
          std::memcpy(&x, &xb, 4);
          if (bits(host_sin(x)) != h[2 * (size_t)i]) {
            s++;
            const int slot = nfs++;
            if (slot < 4) first[slot] = xb;
          }
          if (bits(host_cos(x)) != h[2 * (size_t)i + 1]) {
            c++;
            const int slot = nfc++;
            if (slot < 4) first[4 + slot] = xb;
          }
        }
        ms += s; mc += c;
      });
    for (auto& x : th) x.join();
  }
  cudaFree(d);
  stats[0] = ms; stats[1] = mc; stats[2] = (long long)hi - lo + 1;
  return rc;
}

// the device's and the host's values at one argument: out = {device sin, device cos, host sin, host cos}
int trig_at(float x, float* out) {
  unsigned* d = nullptr;
  if (cudaMalloc(&d, 2 * sizeof(unsigned)) != cudaSuccess) return 1;
  k_trig<<<1, 32>>>(bits(x), 1, d);
  unsigned h[2];
  const int rc = cudaMemcpy(h, d, sizeof h, cudaMemcpyDeviceToHost) != cudaSuccess;
  cudaFree(d);
  std::memcpy(&out[0], &h[0], 4);
  std::memcpy(&out[1], &h[1], 4);
  out[2] = host_sin(x);
  out[3] = host_cos(x);
  return rc;
}

}
