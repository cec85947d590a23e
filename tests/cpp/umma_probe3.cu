// Third UMMA probe (dual build like umma_probe.cu: nvcc for a B200, g++ -DLYRA_EMU for the emulator): the A-operand hand-off
// DecoderKernelDU relies on since it stages the residual units' A operand one k-half at a time in the same TMEM columns.
//   case 9: OUT[128 x 64] = A * W^T in split-precision TF32 with K = 64 and the A operand in TMEM in 2 x 32 columns (hi | lo).
//           The MMAs of channels 0..31 read A, tcgen05.commit arrives on an mbarrier, every thread waits on it and overwrites
//           those A columns with channels 32..63, further MMAs accumulate into the same D.
// A missing wait shows on the hardware as a wrong D.  The emulator executes MMAs at issue, so it cannot catch that; there the
// probe checks the column arithmetic.  Exit code 0 iff the case matches.
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "device_compat.h"

namespace {

constexpr int K = 64, N = 64;

struct HandOffShared { LyraMbar half, done; uint32_t tmem_base; };

__device__ inline int CanonF32(int row, int k, int rows) { return ((k / 4) * (rows / 8) + row / 8) * 32 + (row % 8) * 4 + k % 4; }
__device__ inline void Split(float x, uint32_t& hi, uint32_t& lo) {
  hi = __float_as_uint(x) & 0xffffe000u;
  lo = __float_as_uint(__fsub_rn(x, __uint_as_float(hi)));
}

__global__ void __launch_bounds__(128)
ProbeHandOffKernel(const float* A, const float* W, float* OUT) {
  float* w_hi = reinterpret_cast<float*>(LYRA_DYN_SMEM());
  float* w_lo = w_hi + N * K;
  LYRA_STATIC_SMEM(HandOffShared, sh, 1);
  const int tid = (int)threadIdx.x, warp = tid / 32;
  for (int i = tid; i < N * K; i += 128) {
    uint32_t h, l;
    Split(W[i], h, l);
    w_hi[CanonF32(i / K, i % K, N)] = __uint_as_float(h);
    w_lo[CanonF32(i / K, i % K, N)] = __uint_as_float(l);
  }
  if (tid == 0) { lyra_mbar_init(&sh->half, 1); lyra_mbar_init(&sh->done, 1); lyra_mbar_fence_init(); }
  lyra_fence_proxy_async();
  if (warp == 0) lyra_tmem_alloc(&sh->tmem_base, 128);
  lyra_tc_fence_before_sync();
  __syncthreads();
  lyra_tc_fence_after_sync();
  const uint32_t tmem = sh->tmem_base;
  const uint32_t colAhi = 0, colAlo = 32, colD = 64;
  const uint32_t lane_base = (uint32_t)(32 * warp) << 16;
  for (int h = 0; h < 2; ++h) {
    if (h == 1) {                                   // the MMAs that read channels 0..31 have completed
      lyra_mbar_wait(&sh->half, 0);
      lyra_tc_fence_after_sync();
    }
    for (int c0 = 0; c0 < 32; c0 += 16) {
      uint32_t hi[16], lo[16];
      for (int j = 0; j < 16; ++j) Split(A[tid * K + 32 * h + c0 + j], hi[j], lo[j]);
      lyra_tmem_st<16>(tmem + lane_base + colAhi + (uint32_t)c0, hi);
      lyra_tmem_st<16>(tmem + lane_base + colAlo + (uint32_t)c0, lo);
    }
    lyra_tmem_wait_st();
    lyra_tc_fence_before_sync();
    __syncthreads();
    lyra_tc_fence_after_sync();
    if (tid == 0) {
      const uint32_t idesc = lyra_umma_idesc_tf32(128, N);
      const uint32_t lboW = (uint32_t)(N / 8) * 128u;
      for (int k4 = 0; k4 < 4; ++k4) {
        const int ks = 4 * h + k4;
        const uint64_t bh = lyra_umma_desc(reinterpret_cast<const char*>(w_hi) + (size_t)ks * 2 * lboW, lboW, 128);
        const uint64_t bl = lyra_umma_desc(reinterpret_cast<const char*>(w_lo) + (size_t)ks * 2 * lboW, lboW, 128);
        lyra_umma_tf32_ts(tmem + colD, tmem + colAlo + (uint32_t)(8 * k4), bh, idesc, ks > 0);
        lyra_umma_tf32_ts(tmem + colD, tmem + colAhi + (uint32_t)(8 * k4), bl, idesc, true);
        lyra_umma_tf32_ts(tmem + colD, tmem + colAhi + (uint32_t)(8 * k4), bh, idesc, true);
      }
      lyra_umma_commit(h == 0 ? &sh->half : &sh->done);
    }
  }
  lyra_mbar_wait(&sh->done, 0);
  lyra_tc_fence_after_sync();
  for (int c0 = 0; c0 < N; c0 += 16) {
    uint32_t v[16];
    lyra_tmem_ld<16>(tmem + lane_base + colD + (uint32_t)c0, v);
    lyra_tmem_wait_ld();
    for (int j = 0; j < 16; ++j) OUT[tid * N + c0 + j] = __uint_as_float(v[j]);
  }
  lyra_tc_fence_before_sync();
  __syncthreads();
  if (warp == 0) lyra_tmem_dealloc(tmem, 128);
}

template <typename T>
T* ToDevice(const std::vector<T>& v) {
  void* p = nullptr;
  if (cudaMalloc(&p, v.size() * sizeof(T)) != cudaSuccess) return nullptr;
  cudaMemcpy(p, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice);
  return static_cast<T*>(p);
}

}  // namespace

int main() {
  srand(13);
  auto rnd = [] { return (float)(rand() % 20001 - 10000) / 10000.0f * 1.37f; };
  std::vector<float> A(128 * K), W(N * K), OUT(128 * N);
  for (auto& v : A) v = rnd();
  for (auto& v : W) v = rnd() * 0.25f;
  float *dA = ToDevice(A), *dW = ToDevice(W), *dO = ToDevice(OUT);
  if (!dA || !dW || !dO) { std::printf("allocation failed\n"); return 2; }
  const size_t smem = (size_t)(2 * N * K) * 4;
  LYRA_SET_MAX_SMEM(ProbeHandOffKernel, smem);
  cudaMemset(dO, 0, OUT.size() * 4);
  LYRA_LAUNCH(ProbeHandOffKernel, dim3(1), dim3(128), smem, 0, dA, dW, dO);
  if (cudaDeviceSynchronize() != cudaSuccess) { std::printf("case 9: kernel failed\n"); return 1; }
  cudaMemcpy(OUT.data(), dO, OUT.size() * 4, cudaMemcpyDeviceToHost);
  double worst = 0, scale = 0;
  for (int m = 0; m < 128; ++m)
    for (int n = 0; n < N; ++n) {
      double ref = 0;
      for (int k = 0; k < K; ++k) ref += (double)A[m * K + k] * (double)W[n * K + k];
      worst = std::fmax(worst, std::fabs((double)OUT[m * N + n] - ref));
      scale = std::fmax(scale, std::fabs(ref));
    }
  const bool ok = worst / scale < 5e-6;
  std::printf("case 9 (A k-halves rewritten in TMEM after tcgen05.commit): max |OUT - ref| = %.3e (relative %.2e) -> %s\n",
              worst, worst / scale, ok ? "MATCH" : "MISMATCH");
  return ok ? 0 : 1;
}
