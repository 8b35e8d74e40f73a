// Micro-benchmark of the exponential stream of the attention kernels' softmax / P steps, in registers only (no TMEM, no
// barriers): how many cycles does a warp need per 64-element half-row when the exponentials go to the MUFU pipe, to
// the FMA pipe (exp2_poly2), or to a mix -- with one warp per SM sub-partition (what a ping-pong kernel has while the
// other tile waits for the tensor pipe) and with two (both tiles' warps in their exp phase at once).
//   variant 0: 64 x ex2 only (the MUFU pipe's cadence as one warp sees it)
//   variant 1: production pattern: x = s * scale - m (FFMA2), ex2 x 2, row sum (FADD2), 16-bit pack (F2FP)
//   variant 2: same through softmax_exp_half (in place, skewed)
//   variant 3: x pair -> f16x2 (F2FP), ONE ex2.approx.ftz.f16x2 per pair; the result IS the packed FP16 P (no row sum:
//              l would come from a ones column of V on the tensor core)
//   variant 4: variant 3 plus an FP32 row sum of the unpacked results
// each with kPoly = 0..4 of every 4 pairs on the FMA pipe (variant 0: ignored).
// Build: make -C tests/gpu_probe   Run (GPU box): tests/gpu_probe/_build/exp_probe
#include <cstdio>
#include <cstdlib>
#include <vector>

#include "sm100_ptx.cuh"

using namespace mfa::ptx;

template <int VARIANT, int POLY>
__device__ __forceinline__ float step(float (&s)[64], uint32_t (&packed)[32], float scale_log2, float m) {
  if (VARIANT == 0) {
    float acc0 = 0.f, acc1 = 0.f;
#pragma unroll
    for (uint32_t i = 0; i < 32; ++i) {
      s[2 * i] = ex2_approx(s[2 * i]);
      s[2 * i + 1] = ex2_approx(s[2 * i + 1]);
    }
#pragma unroll
    for (uint32_t i = 0; i < 32; ++i) {
      acc0 += s[2 * i];
      acc1 += s[2 * i + 1];
      s[2 * i] = s[2 * i] * 0.25f - 1.0f;  // keep the values bounded for the next round
      s[2 * i + 1] = s[2 * i + 1] * 0.25f - 1.0f;
    }
    return acc0 + acc1;
  } else if (VARIANT == 1) {
    float2 sum2 = make_float2(0.f, 0.f);
    const float2 scale2 = make_float2(scale_log2, scale_log2), negm2 = make_float2(-m, -m);
#pragma unroll
    for (uint32_t i = 0; i < 32; ++i) {
      const float2 x = ffma2(make_float2(s[2 * i], s[2 * i + 1]), scale2, negm2);
      float2 pr;
      if (POLY > 0 && (i & 3) < POLY) {
        pr = exp2_poly2(x);
      } else {
        pr.x = ex2_approx(x.x);
        pr.y = ex2_approx(x.y);
      }
      sum2 = fadd2(sum2, pr);
      packed[i] = pack_bf16x2(pr.x, pr.y);
    }
    return sum2.x + sum2.y;
  } else if (VARIANT == 2) {
    uint32_t v[64];
#pragma unroll
    for (uint32_t i = 0; i < 64; ++i) v[i] = __float_as_uint(s[i]);
    return softmax_exp_half<true, POLY>(v, packed, scale_log2, m);
  } else {
    float2 sum2 = make_float2(0.f, 0.f);
    const float2 scale2 = make_float2(scale_log2, scale_log2), negm2 = make_float2(-m, -m);
#pragma unroll
    for (uint32_t i = 0; i < 32; ++i) {
      const float2 x = ffma2(make_float2(s[2 * i], s[2 * i + 1]), scale2, negm2);
      const uint32_t xh = pack_f16x2(x.x, x.y);
      uint32_t ph;
      asm volatile("ex2.approx.f16x2 %0, %1;" : "=r"(ph) : "r"(xh));
      packed[i] = ph;
      if (VARIANT == 4) sum2 = fadd2(sum2, unpack_f16x2(ph));
    }
    return sum2.x + sum2.y;
  }
}

template <int VARIANT, int POLY>
__global__ void __launch_bounds__(256, 1) exp_probe(float *sink, long long *cycles, int iters, float scale_log2, float m) {
  float s[64];
#pragma unroll
  for (uint32_t i = 0; i < 64; ++i) {
    uint32_t h = (threadIdx.x * 131u + i * 2654435761u) ^ (blockIdx.x * 97u);
    h ^= h >> 13;
    h *= 0x5bd1e995u;
    h ^= h >> 15;
    s[i] = (static_cast<float>(h & 0xffff) / 65536.0f - 0.5f) * 6.0f;
  }
  float l = 0.f;
  uint32_t x = 0;
  __syncthreads();
  const long long t0 = clock64();
  for (int it = 0; it < iters; ++it) {
    uint32_t packed[32];
#pragma unroll
    for (uint32_t i = 0; i < 32; ++i) packed[i] = 0;
    l += step<VARIANT, POLY>(s, packed, scale_log2, m);
#pragma unroll
    for (uint32_t i = 0; i < 32; ++i) x ^= packed[i];
    if (VARIANT != 0) {
      // perturb the inputs so that no round can be hoisted; one FMA-pipe instruction per pair, like the FFMA2 above
      const float d = __uint_as_float((x & 1u) << 20);
#pragma unroll
      for (uint32_t i = 0; i < 64; i += 2) {
        const float2 t = fadd2(make_float2(s[i], s[i + 1]), make_float2(d, d));
        s[i] = t.x;
        s[i + 1] = t.y;
      }
    }
  }
  const long long t1 = clock64();
  sink[blockIdx.x * blockDim.x + threadIdx.x] = l + __uint_as_float(x & 0x3fffffu);
  if ((threadIdx.x & 31) == 0) cycles[blockIdx.x * (blockDim.x / 32) + threadIdx.x / 32] = t1 - t0;
}

template <int VARIANT, int POLY>
static void run(const char *name, int warps) {
  const int ctas = 148, iters = 4000, threads = warps * 32;
  float *sink;
  long long *cycles;
  cudaMalloc(&sink, ctas * threads * sizeof(float));
  cudaMalloc(&cycles, ctas * warps * sizeof(long long));
  auto kernel = exp_probe<VARIANT, POLY>;
  for (int rep = 0; rep < 2; ++rep) kernel<<<ctas, threads>>>(sink, cycles, iters, 0.1275f, 0.5f);
  cudaError_t e = cudaDeviceSynchronize();
  if (e != cudaSuccess) {
    printf("%s: CUDA error %s\n", name, cudaGetErrorString(e));
    exit(1);
  }
  std::vector<long long> h(ctas * warps);
  cudaMemcpy(h.data(), cycles, h.size() * sizeof(long long), cudaMemcpyDeviceToHost);
  double sum = 0;
  for (long long c : h) sum += static_cast<double>(c);
  const double per_half = sum / h.size() / iters;
  printf("%-44s poly %d/4  %d warp(s)/sub-partition: %6.0f cycles per 64-element half-row per warp = %5.2f cycles per "
         "element pair; SM-wide %5.1f exp/clk\n",
         name, POLY, warps / 4, per_half, per_half / 32, 64.0 * 32 * warps / per_half);
  cudaFree(sink);
  cudaFree(cycles);
}

template <int VARIANT, int POLY>
static void both(const char *name) {
  run<VARIANT, POLY>(name, 4);
  run<VARIANT, POLY>(name, 8);
}

int main() {
  both<0, 0>("ex2 only");
  both<1, 0>("production loop (scale, ex2, sum, pack)");
  both<1, 1>("production loop (scale, ex2, sum, pack)");
  both<1, 2>("production loop (scale, ex2, sum, pack)");
  both<1, 3>("production loop (scale, ex2, sum, pack)");
  both<1, 4>("production loop (scale, ex2, sum, pack)");
  both<2, 0>("softmax_exp_half (in place, skewed)");
  both<2, 1>("softmax_exp_half (in place, skewed)");
  both<2, 2>("softmax_exp_half (in place, skewed)");
  both<3, 0>("f16x2 ex2 (one MUFU per pair), no row sum");
  both<4, 0>("f16x2 ex2 (one MUFU per pair) + FP32 row sum");
  return 0;
}
