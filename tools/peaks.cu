// tools/peaks.cu -- measured denominators that MEASURED_PEAKS.json does not carry (VERDICT r1 item 9):
//   * FP32 FFMA throughput of the CUDA cores (the roofline of the FP32 half-step kernel, nominally 148 x 128 x 2 x f),
//   * mma.sync m16n8k8 TF32 and m16n8k16 FP16 (f32 accumulate) throughput (the warp-level tensor paths; the rank-64 pair
//     kernel accumulates on the FP16 one),
//   * warp shuffle and shared-memory LDS.128 issue rates (the other two pipes the solve leans on).
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -o tools/peaks tools/peaks.cu ; run on the GPU box, prints JSON.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#define CK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { fprintf(stderr, "%s: %s\n", #x, cudaGetErrorString(e_)); return 1; } } while (0)

__global__ void __launch_bounds__(256) ffma_kernel(float* out, int iters, float x, float y) {
  float a[16];
#pragma unroll
  for (int j = 0; j < 16; ++j) a[j] = (float)(threadIdx.x + j);
#pragma unroll 1
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int r = 0; r < 8; ++r)
#pragma unroll
      for (int j = 0; j < 16; ++j) a[j] = fmaf(a[j], x, y);
  }
  float s = 0.f;
#pragma unroll
  for (int j = 0; j < 16; ++j) s += a[j];
  out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}

__global__ void __launch_bounds__(256) mma_kernel(float* out, int iters) {
  float d[8][4];
#pragma unroll
  for (int j = 0; j < 8; ++j)
#pragma unroll
    for (int e = 0; e < 4; ++e) d[j][e] = 0.f;
  uint32_t a[4] = {threadIdx.x, threadIdx.x + 1u, threadIdx.x + 2u, threadIdx.x + 3u};
  uint32_t b0 = threadIdx.x * 3u, b1 = threadIdx.x * 5u;
#pragma unroll 1
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int j = 0; j < 8; ++j)
      asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};\n"
                   : "+f"(d[j][0]), "+f"(d[j][1]), "+f"(d[j][2]), "+f"(d[j][3])
                   : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
  }
  float s = 0.f;
#pragma unroll
  for (int j = 0; j < 8; ++j) s += d[j][0] + d[j][1] + d[j][2] + d[j][3];
  out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}

__global__ void __launch_bounds__(256) mma_k4_kernel(float* out, int iters) {
  float d[8][4];
#pragma unroll
  for (int j = 0; j < 8; ++j)
#pragma unroll
    for (int e = 0; e < 4; ++e) d[j][e] = 0.f;
  uint32_t a[2] = {threadIdx.x, threadIdx.x + 1u};
  uint32_t b0 = threadIdx.x * 3u;
#pragma unroll 1
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int j = 0; j < 8; ++j)
      asm volatile("mma.sync.aligned.m16n8k4.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5}, {%6}, {%0,%1,%2,%3};\n"
                   : "+f"(d[j][0]), "+f"(d[j][1]), "+f"(d[j][2]), "+f"(d[j][3])
                   : "r"(a[0]), "r"(a[1]), "r"(b0));
  }
  float s = 0.f;
#pragma unroll
  for (int j = 0; j < 8; ++j) s += d[j][0] + d[j][1] + d[j][2] + d[j][3];
  out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}

__global__ void __launch_bounds__(256) mma_f16_kernel(float* out, int iters) {
  float d[8][4];
#pragma unroll
  for (int j = 0; j < 8; ++j)
#pragma unroll
    for (int e = 0; e < 4; ++e) d[j][e] = 0.f;
  uint32_t a[4] = {threadIdx.x, threadIdx.x + 1u, threadIdx.x + 2u, threadIdx.x + 3u};
  uint32_t b0 = threadIdx.x * 3u, b1 = threadIdx.x * 5u;
#pragma unroll 1
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int j = 0; j < 8; ++j)
      asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};\n"
                   : "+f"(d[j][0]), "+f"(d[j][1]), "+f"(d[j][2]), "+f"(d[j][3])
                   : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
  }
  float s = 0.f;
#pragma unroll
  for (int j = 0; j < 8; ++j) s += d[j][0] + d[j][1] + d[j][2] + d[j][3];
  out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}

__global__ void __launch_bounds__(256) shfl_kernel(float* out, int iters) {
  float v[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) v[j] = (float)(threadIdx.x * 8 + j);
#pragma unroll 1
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = __shfl_sync(0xffffffffu, v[j], (threadIdx.x + j + 1) & 31);
  }
  float s = 0.f;
#pragma unroll
  for (int j = 0; j < 8; ++j) s += v[j];
  out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}

__global__ void __launch_bounds__(256) lds_kernel(float* out, int iters) {
  __shared__ __align__(16) float sm[256 * 4 * 2];
  for (int o = threadIdx.x; o < 2048; o += 256) sm[o] = (float)o;
  __syncthreads();
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  const float4* p = reinterpret_cast<const float4*>(sm);
  int idx = threadIdx.x;
#pragma unroll 1
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float4 v = p[(idx + j * 32) & 511];
      acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
    }
    idx = (idx + 7) & 511;
  }
  out[blockIdx.x * blockDim.x + threadIdx.x] = acc.x + acc.y + acc.z + acc.w;
}

// fp64: the scoring kernels accumulate in double like the JVM (bit-exact top-k), so their compute bound is the DFMA pipe
__global__ void __launch_bounds__(256) dfma_kernel(float* out, int iters, double x, double y) {
  double a[16];
#pragma unroll
  for (int j = 0; j < 16; ++j) a[j] = (double)(threadIdx.x + j);
#pragma unroll 1
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int r = 0; r < 8; ++r)
#pragma unroll
      for (int j = 0; j < 16; ++j) a[j] = fma(a[j], x, y);
  }
  double s = 0.0;
#pragma unroll
  for (int j = 0; j < 16; ++j) s += a[j];
  out[blockIdx.x * blockDim.x + threadIdx.x] = (float)s;
}
// float -> double conversions (F2F.F64.F32, one per matrix element scored)
__global__ void __launch_bounds__(256) f2f_kernel(float* out, int iters, float x) {
  float a[16];
#pragma unroll
  for (int j = 0; j < 16; ++j) a[j] = (float)(threadIdx.x + j) * x;
  int acc = 0;
#pragma unroll 1
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int r = 0; r < 4; ++r)
#pragma unroll
      for (int j = 0; j < 16; ++j) {
        acc ^= __double2hiint((double)a[j]);   // one F2F.F64.F32 per element; the XOR and the FMUL run on other pipes
        a[j] *= x;
      }
  }
  out[blockIdx.x * blockDim.x + threadIdx.x] = (float)acc + a[3];
}

int main() {
  cudaDeviceProp pr;
  CK(cudaGetDeviceProperties(&pr, 0));
  const int sms = pr.multiProcessorCount;
  const int blocks = sms * 8, threads = 256;
  float* out = nullptr;
  CK(cudaMalloc(&out, sizeof(float) * blocks * threads));
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0);
  cudaEventCreate(&e1);
  float ms = 0.f, best;
  double ffma_tf = 0, mma_tf = 0, shfl_rate = 0, lds_bpc = 0;
  const int iters = 4000;
  // FFMA
  best = 1e30f;
  for (int rep = 0; rep < 5; ++rep) {
    cudaEventRecord(e0);
    ffma_kernel<<<blocks, threads>>>(out, iters, 1.0001f, 0.5f);
    cudaEventRecord(e1);
    CK(cudaDeviceSynchronize());
    cudaEventElapsedTime(&ms, e0, e1);
    if (rep > 0 && ms < best) best = ms;
  }
  ffma_tf = 2.0 * 16 * 8 * (double)iters * blocks * threads / (best * 1e-3) / 1e12;
  const double ffma_ms = best;
  // mma.sync tf32
  best = 1e30f;
  for (int rep = 0; rep < 5; ++rep) {
    cudaEventRecord(e0);
    mma_kernel<<<blocks, threads>>>(out, iters);
    cudaEventRecord(e1);
    CK(cudaDeviceSynchronize());
    cudaEventElapsedTime(&ms, e0, e1);
    if (rep > 0 && ms < best) best = ms;
  }
  mma_tf = 2.0 * 16 * 8 * 8 * 8.0 * (double)iters * blocks * (threads / 32) / (best * 1e-3) / 1e12;
  const double mma_per_sm_clk = 8.0 * (double)iters * blocks * (threads / 32) / sms / (best * 1e-3 * pr.clockRate * 1e3);
  // mma.sync tf32 k4
  best = 1e30f;
  for (int rep = 0; rep < 5; ++rep) {
    cudaEventRecord(e0);
    mma_k4_kernel<<<blocks, threads>>>(out, iters);
    cudaEventRecord(e1);
    CK(cudaDeviceSynchronize());
    cudaEventElapsedTime(&ms, e0, e1);
    if (rep > 0 && ms < best) best = ms;
  }
  const double mma4_per_sm_clk = 8.0 * (double)iters * blocks * (threads / 32) / sms / (best * 1e-3 * pr.clockRate * 1e3);
  // mma.sync f16 k16, f32 accumulate
  best = 1e30f;
  for (int rep = 0; rep < 5; ++rep) {
    cudaEventRecord(e0);
    mma_f16_kernel<<<blocks, threads>>>(out, iters);
    cudaEventRecord(e1);
    CK(cudaDeviceSynchronize());
    cudaEventElapsedTime(&ms, e0, e1);
    if (rep > 0 && ms < best) best = ms;
  }
  const double mma16_tf = 2.0 * 16 * 8 * 16 * 8.0 * (double)iters * blocks * (threads / 32) / (best * 1e-3) / 1e12;
  const double mma16_per_sm_clk = 8.0 * (double)iters * blocks * (threads / 32) / sms / (best * 1e-3 * pr.clockRate * 1e3);
  // shfl
  best = 1e30f;
  for (int rep = 0; rep < 5; ++rep) {
    cudaEventRecord(e0);
    shfl_kernel<<<blocks, threads>>>(out, iters);
    cudaEventRecord(e1);
    CK(cudaDeviceSynchronize());
    cudaEventElapsedTime(&ms, e0, e1);
    if (rep > 0 && ms < best) best = ms;
  }
  shfl_rate = 8.0 * (double)iters * blocks * (threads / 32) / sms / (best * 1e-3 * pr.clockRate * 1e3);
  // LDS.128
  best = 1e30f;
  for (int rep = 0; rep < 5; ++rep) {
    cudaEventRecord(e0);
    lds_kernel<<<blocks, threads>>>(out, iters);
    cudaEventRecord(e1);
    CK(cudaDeviceSynchronize());
    cudaEventElapsedTime(&ms, e0, e1);
    if (rep > 0 && ms < best) best = ms;
  }
  lds_bpc = 8.0 * 512.0 * (double)iters * blocks * (threads / 32) / sms / (best * 1e-3 * pr.clockRate * 1e3);
  // DFMA
  best = 1e30f;
  const int diters = 400;
  for (int rep = 0; rep < 5; ++rep) {
    cudaEventRecord(e0);
    dfma_kernel<<<blocks, threads>>>(out, diters, 1.0000001, 0.5);
    cudaEventRecord(e1);
    CK(cudaDeviceSynchronize());
    cudaEventElapsedTime(&ms, e0, e1);
    if (rep > 0 && ms < best) best = ms;
  }
  const double dfma_tf = 2.0 * 16 * 8 * (double)diters * blocks * threads / (best * 1e-3) / 1e12;
  const double dfma_per_sm_clk = 16.0 * 8 * (double)diters * blocks * threads / sms / (best * 1e-3 * pr.clockRate * 1e3);
  // F2F.F64.F32
  best = 1e30f;
  for (int rep = 0; rep < 5; ++rep) {
    cudaEventRecord(e0);
    f2f_kernel<<<blocks, threads>>>(out, diters, 1.5f);
    cudaEventRecord(e1);
    CK(cudaDeviceSynchronize());
    cudaEventElapsedTime(&ms, e0, e1);
    if (rep > 0 && ms < best) best = ms;
  }
  const double f2f_per_sm_clk = 4.0 * 16 * (double)diters * blocks * threads / sms / (best * 1e-3 * pr.clockRate * 1e3);
  printf("{\"gpu\": \"%s\", \"sms\": %d, \"clock_mhz_max\": %.0f, \"ffma_tflops\": %.2f, \"ffma_ms\": %.3f, "
         "\"ffma_nominal_tflops\": %.2f, \"mma_sync_tf32_tflops\": %.2f, \"mma_sync_m16n8k8_per_sm_per_clk_at_max_clock\": %.4f, "
         "\"mma_sync_m16n8k4_per_sm_per_clk_at_max_clock\": %.4f, "
         "\"mma_sync_f16_m16n8k16_tflops\": %.2f, \"mma_sync_f16_m16n8k16_per_sm_per_clk_at_max_clock\": %.4f, \"shfl_warp_instr_per_sm_per_clk_at_max_clock\": %.3f, \"lds128_bytes_per_sm_per_clk_at_max_clock\": %.1f, "
         "\"dfma_tflops\": %.2f, \"dfma_lanes_per_sm_per_clk_at_max_clock\": %.2f, \"f2f_f64_f32_lanes_per_sm_per_clk_at_max_clock\": %.2f, "
         "\"how\": \"tools/peaks.cu: 8 CTAs x 256 threads per SM, best of 4 timed launches, CUDA events\"}\n",
         pr.name, sms, pr.clockRate / 1e3, ffma_tf, ffma_ms, sms * 128 * 2 * (pr.clockRate * 1e3) / 1e12, mma_tf,
         mma_per_sm_clk, mma4_per_sm_clk, mma16_tf, mma16_per_sm_clk, shfl_rate, lds_bpc, dfma_tf, dfma_per_sm_clk, f2f_per_sm_clk);
  return 0;
}
