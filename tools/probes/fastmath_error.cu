// How far are the intrinsics of the in-kernel Box-Muller (common.cuh, philox_normal4) from the exact functions, over
// every argument that kernel can give them?  Exhaustive over float32 bit patterns, double-precision reference:
//   __sincosf on [0, 6.2831855f]: the kernel's angle (float)(2 pi) * u with u in (0, 1] — beyond the [-pi, pi] the CUDA
//     programming guide documents;
//   __logf on [2^-33, 1]: the uniforms u32_to_uniform produces; absolute error on [0.5, 1], ulp error below 0.5.
// tests/test_gpu_noise_streams.py takes its __sincosf term from this measurement.
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -o fastmath_error fastmath_error.cu && ./fastmath_error
#include <cstdio>
#include <cstring>
#include <cuda_runtime.h>

__device__ void atomic_max_pos(unsigned long long* p, double v) {   // non-negative doubles order as their bit patterns
  atomicMax(p, (unsigned long long)__double_as_longlong(v));
}

__global__ void sincos_err(unsigned lo_bits, unsigned hi_bits, unsigned long long* out) {
  double es = 0.0, ec = 0.0;
  for (unsigned long long b = lo_bits + blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; b <= hi_bits;
       b += (unsigned long long)gridDim.x * blockDim.x) {
    const float x = __uint_as_float((unsigned)b);
    float s, c;
    __sincosf(x, &s, &c);
    double sr, cr;
    sincos((double)x, &sr, &cr);
    es = fmax(es, fabs((double)s - sr));
    ec = fmax(ec, fabs((double)c - cr));
  }
  atomic_max_pos(out + 0, es);
  atomic_max_pos(out + 1, ec);
}

__global__ void log_err(unsigned lo_bits, unsigned hi_bits, unsigned long long* out) {
  double eabs = 0.0, eulp = 0.0;
  for (unsigned long long b = lo_bits + blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; b <= hi_bits;
       b += (unsigned long long)gridDim.x * blockDim.x) {
    const float x = __uint_as_float((unsigned)b);
    const double r = log((double)x), e = fabs((double)__logf(x) - r);
    if (x >= 0.5f) {
      eabs = fmax(eabs, e);
    } else {
      int ex;
      frexp(r, &ex);
      eulp = fmax(eulp, e / ldexp(1.0, ex - 24));   // ulp of a float in [2^(ex-1), 2^ex)
    }
  }
  atomic_max_pos(out + 2, eabs);
  atomic_max_pos(out + 3, eulp);
}

static unsigned bits(float f) { unsigned u; memcpy(&u, &f, 4); return u; }

int main() {
  cudaDeviceProp prop;
  cudaGetDeviceProperties(&prop, 0);
  unsigned long long* d;
  cudaMalloc(&d, 4 * sizeof(unsigned long long));
  cudaMemset(d, 0, 4 * sizeof(unsigned long long));
  sincos_err<<<4096, 256>>>(0u, bits(6.283185307179586f), d);
  log_err<<<4096, 256>>>(bits(0x1p-33f), bits(1.0f), d);
  unsigned long long h[4];
  cudaError_t e = cudaMemcpy(h, d, sizeof(h), cudaMemcpyDeviceToHost);
  if (e != cudaSuccess) { printf("error: %s\n", cudaGetErrorString(e)); return 1; }
  double v[4];
  memcpy(v, h, sizeof(v));
  printf("device %s\n", prop.name);
  printf("__sincosf on [0, 2pi]: max abs error sin %.4g (2^%.2f), cos %.4g (2^%.2f)\n", v[0], log2(v[0]), v[1], log2(v[1]));
  printf("__logf on [0.5, 1]: max abs error %.4g (2^%.2f); on [2^-33, 0.5): max error %.3g ulp\n", v[2], log2(v[2]), v[3]);
  cudaFree(d);
  return 0;
}
