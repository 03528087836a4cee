// Probe: is the fp32 accumulator of tcgen05.mma.kind::f16 exact for integer-valued fp16 operands?
// conv1_tc.cu feeds the tensor core A = x - zp_x in [-255, 255] and B = w in [-128, 127] and uses the fp32 accumulator
// as f32(acc - corr).  Every product is an integer below 2^15 and every partial sum of its 27 (here up to 48) terms an
// integer below 2^24, so the result must be exact in any summation order.  This runs M=128, N=64, K=16 MMAs chained 1,
// 2 and 3 deep into one accumulator (SWIZZLE_32B K-major operands, the layout of conv1_tc.cu) and compares every output
// against int64 host sums.
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -o probe_f16_intacc tools/probe_f16_intacc.cu
#include <cstdio>
#include <algorithm>
#include <cstdint>
#include <cstring>
#include <random>
#include <vector>
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include "../convnet_quantization_b200/csrc/common.cuh"
namespace b200q { void set_error(const char*, ...) {} int check_cuda(cudaError_t, const char*) { return 0; } int launched(const char*) { return 0; } int num_sms() { return 148; }
int encode_tensor_map(CUtensorMap*, const void*, int, const uint64_t*, const uint64_t*, const uint32_t*, int) { return 0; } }
using namespace b200q;

constexpr int M = 128, N = 64, K = 16, MAXCHAIN = 3;

__device__ __forceinline__ uint32_t swz32(uint32_t lin) { return lin ^ (((lin >> 7) & 1) << 4); }

// a: [chain][M][K], b: [chain][N][K] integers; out: [M][N] fp32 bits
__global__ void __launch_bounds__(128, 1) intacc_probe(const int16_t* a, const int16_t* b, int chain, uint32_t* out) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* sa = smem;                        // [chain][M][32 B]
  uint8_t* sb = smem + MAXCHAIN * M * 32;    // [chain][N][32 B]
  __shared__ uint64_t bar;
  __shared__ uint32_t tmem_base_s;
  for (int i = threadIdx.x; i < chain * M * K; i += blockDim.x) {
    const int c = i / (M * K), r = (i / K) % M, k = i % K;
    *reinterpret_cast<__half*>(sa + c * M * 32 + swz32(r * 32 + k * 2)) = __int2half_rn(a[i]);
  }
  for (int i = threadIdx.x; i < chain * N * K; i += blockDim.x) {
    const int c = i / (N * K), r = (i / K) % N, k = i % K;
    *reinterpret_cast<__half*>(sb + c * N * 32 + swz32(r * 32 + k * 2)) = __int2half_rn(b[i]);
  }
  if (threadIdx.x == 0) { mbar_init(&bar, 1); fence_barrier_init(); }
  if (threadIdx.x < 32) { tmem_alloc(&tmem_base_s, 64); tmem_relinquish(); }
  fence_proxy_async_smem();
  tc_fence_before(); __syncthreads(); tc_fence_after();
  const uint32_t tmem = tmem_base_s;
  if (threadIdx.x == 0) {
    constexpr uint32_t idesc = make_idesc_f16(M, N);
    for (int c = 0; c < chain; ++c)
      tc_mma_f16(tmem, make_kmajor_desc<32>(smem_u32(sa + c * M * 32), 256), make_kmajor_desc<32>(smem_u32(sb + c * N * 32), 256),
                 idesc, c > 0 ? 1u : 0u);
    tc_commit(&bar);
    mbar_wait(&bar, 0);
  }
  __syncthreads();
  tc_fence_after();
  const int warp = threadIdx.x >> 5;
  for (int half = 0; half < 2; ++half) {
    uint32_t v[32];
    tmem_ld_32x32(tmem + ((uint32_t)(warp * 32) << 16) + half * 32, v);
    tmem_ld_wait();
    for (int j = 0; j < 32; ++j) out[threadIdx.x * N + half * 32 + j] = v[j];
  }
  tc_fence_before(); __syncthreads();
  if (threadIdx.x < 32) tmem_dealloc(tmem, 64);
}

int main() {
  int16_t *d_a, *d_b; uint32_t* d_out;
  cudaMalloc(&d_a, MAXCHAIN * M * K * 2); cudaMalloc(&d_b, MAXCHAIN * N * K * 2); cudaMalloc(&d_out, M * N * 4);
  const int smem = MAXCHAIN * (M + N) * 32 + 1024;
  cudaFuncSetAttribute(intacc_probe, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
  std::mt19937 rng(12345);
  std::vector<int16_t> a(MAXCHAIN * M * K), b(MAXCHAIN * N * K);
  std::vector<uint32_t> h(M * N);
  long total_bad = 0, total = 0;
  const char* names[] = {"all +255 x +127", "all -255 x -128", "all +255 x -128", "cancel then small", "random"};
  for (int cs = 0; cs < 5; ++cs)
    for (int chain = 1; chain <= MAXCHAIN; ++chain) {
      for (int c = 0; c < MAXCHAIN; ++c) {
        for (int r = 0; r < M; ++r)
          for (int k = 0; k < K; ++k) {
            int16_t& x = a[(c * M + r) * K + k];
            if (cs == 0 || cs == 2) x = 255;
            else if (cs == 1) x = -255;
            else if (cs == 3) x = (c == 0) ? (k < 8 ? 255 : -255) : (k < 8 ? -255 : (int16_t)((r + k) % 7 - 3));
            else x = (int16_t)((int)(rng() % 511) - 255);
          }
        for (int n = 0; n < N; ++n)
          for (int k = 0; k < K; ++k) {
            int16_t& w = b[(c * N + n) * K + k];
            if (cs == 0) w = 127;
            else if (cs == 1 || cs == 2) w = -128;
            // large same-sign products in the first MMA, a near-cancelling second, small terms after
            else if (cs == 3) w = (c == 0) ? (k < 8 ? -128 : 127) : (k < 8 ? ((n & 1) ? -128 : 127) : (int16_t)((n + k) % 5 - 2));
            else w = (int16_t)((int)(rng() % 256) - 128);
          }
      }
      cudaMemcpy(d_a, a.data(), a.size() * 2, cudaMemcpyHostToDevice);
      cudaMemcpy(d_b, b.data(), b.size() * 2, cudaMemcpyHostToDevice);
      intacc_probe<<<1, 128, smem>>>(d_a, d_b, chain, d_out);
      const cudaError_t e = cudaDeviceSynchronize();
      if (e != cudaSuccess) { printf("%s chain %d: %s\n", names[cs], chain, cudaGetErrorString(e)); return 1; }
      cudaMemcpy(h.data(), d_out, h.size() * 4, cudaMemcpyDeviceToHost);
      int bad = 0;
      int64_t maxabs = 0;
      for (int r = 0; r < M; ++r)
        for (int n = 0; n < N; ++n) {
          int64_t ref = 0;
          for (int c = 0; c < chain; ++c)
            for (int k = 0; k < K; ++k) ref += (int64_t)a[(c * M + r) * K + k] * b[(c * N + n) * K + k];
          float got;
          memcpy(&got, &h[r * N + n], 4);
          maxabs = std::max(maxabs, ref < 0 ? -ref : ref);
          if ((double)got != (double)ref) {
            if (bad < 4) printf("  mismatch row %d col %d: got %.1f want %lld\n", r, n, got, (long long)ref);
            ++bad;
          }
        }
      printf("%-18s chain %d: %d / %d mismatches (max |sum| %lld)\n", names[cs], chain, bad, M * N, (long long)maxabs);
      total_bad += bad;
      total += M * N;
    }
  printf("TOTAL: %ld mismatches of %ld outputs\n", total_bad, total);
  return total_bad != 0;
}
