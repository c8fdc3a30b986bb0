// Throughput of two fp64 tanh for the epilogue of a basis layer on the FP64 pipe: libdevice tanh(), which the library uses,
// against the table-driven candidate below.  Every thread runs a dependent chain x <- 3 tanh(x) + c over its own element,
// with the inputs spread over [-4, 4] so that warps take both branches of each implementation, as a layer's pre-activations
// do.  Prints one JSON line.  Built and run by tools/dngo_act.py (DESIGN.md section 4.5 has the result).
#include <cstdio>
#include <vector>

#include "../bot7_b200/csrc/exp_neg.cuh"

// The candidate, reusing exp_neg.cuh's table-driven exp(x <= 0):
//   |x| <  0.625: x + x^3 Q(x^2), Q of degree 11 fitted for relative error (6.8e-17 on [0, 0.390625]);
//   |x| >= 0.625: (1 - e) / (1 + e), e = exp_neg(-2|x|); from 0.625 on the error of e reaches the quotient scaled by
//                 2e / (1 - e^2) <= 0.63, below it 1 - e cancels, hence the polynomial;
// then the sign of x.  Worst error seen against mpmath on 2e5 points over [1e-300, 800]: 1.70 ulp.  e = 0 for |x| > 354 gives
// exactly 1 (+-inf -> +-1), NaN stays NaN.
__device__ __forceinline__ double b7_tanh(double x) {
  const double t = fabs(x);
  double y;
  if (t < 0.625) {
    const double u = t * t;
    double q = 6.476658369354856e-06;
    q = fma(q, u, -3.118276779963142e-05);
    q = fma(q, u, 9.255408976445487e-05);
    q = fma(q, u, -0.0002375816628927853);
    q = fma(q, u, 0.0005896577189384784);
    q = fma(q, u, -0.0014557747943454275);
    q = fma(q, u, 0.003592121667721315);
    q = fma(q, u, -0.008863235096209671);
    q = fma(q, u, 0.021869488518662286);
    q = fma(q, u, -0.05396825396788825);
    q = fma(q, u, 0.13333333333333033);
    q = fma(q, u, -0.3333333333333333);
    y = fma(t * u, q, t);
  } else {
    const double e = exp_neg(-2.0 * t, c_exp_tab);
    y = (1.0 - e) / (1.0 + e);
  }
  return copysign(y, x);
}

template <int F>
__global__ void chain(double* x, long long n, int reps) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double v = x[i];
  const double c = 0.25 * (double)(i & 7) - 0.9;
  for (int r = 0; r < reps; ++r) v = fma(3.0, F ? tanh(v) : b7_tanh(v), c);
  x[i] = v;
}

int main() {
  const long long n = 1LL << 24;
  const int reps = 32, iters = 20;
  std::vector<double> h(n);
  for (long long i = 0; i < n; ++i) h[i] = -4.0 + 8.0 * (double)((i * 2654435761LL) % 1000003) / 1000003.0;
  double* d;
  cudaMalloc(&d, n * 8);
  cudaEvent_t a, b;
  cudaEventCreate(&a);
  cudaEventCreate(&b);
  float ms[2] = {0.f, 0.f};
  for (int round = 0; round < 2; ++round)              // round 0 warms both kernels up
    for (int f = 0; f < 2; ++f) {
      cudaMemcpy(d, h.data(), n * 8, cudaMemcpyHostToDevice);
      cudaEventRecord(a);
      for (int it = 0; it < iters; ++it) {
        if (f) chain<1><<<(unsigned)(n / 256), 256>>>(d, n, reps);
        else chain<0><<<(unsigned)(n / 256), 256>>>(d, n, reps);
      }
      cudaEventRecord(b);
      cudaEventSynchronize(b);
      if (round) cudaEventElapsedTime(&ms[f], a, b);
    }
  if (cudaGetLastError() != cudaSuccess) { fprintf(stderr, "tanh_bench: CUDA error\n"); return 1; }
  const double evals = (double)n * reps * iters;
  printf("{\"evals\": %.0f, \"b7_tanh_ns_per_1k\": %.4f, \"libdevice_tanh_ns_per_1k\": %.4f}\n", evals, ms[0] * 1e9 / evals,
         ms[1] * 1e9 / evals);
  cudaFree(d);
  return 0;
}
