// ensemble.cu -- per-pixel statistics of an ensemble of N super-resolved fields (wsr_ensemble_stats): mean and spread fields, the
// per-plane sums behind CRPS (standard and fair), the spread-skill ratio and the rank histogram.  One thread owns one pixel and
// reads its N member values (member-major input: consecutive threads read consecutive addresses of one member row), sorts them,
// and accumulates in double.  Sorting: a bitonic network in registers for N <= 8, a per-thread column of shared memory
// (s[k * blockDim + tid], conflict-free) for 8 < N <= 256 (a 16- or 32-wide register network needs 155 / 255 registers).  Block partial sums go through shared memory; one atomic per
// (plane, quantity) and per non-empty histogram bin per block.
#include "common.cuh"

namespace wsr {

constexpr int kEnsK = 5;             // accumulator quantities per plane (wsr.h)

__device__ __forceinline__ void cswap(float& a, float& b) {
  const float lo = fminf(a, b), hi = fmaxf(a, b);
  a = lo; b = hi;
}

// Per-pixel contribution from the N sorted member values v(k), k < N, and the target y.
struct PixelAcc {
  double q[kEnsK];
  __device__ void zero() {
#pragma unroll
    for (int k = 0; k < kEnsK; ++k) q[k] = 0.0;
  }
};

// LOOP: compile-time bound of k (the register path unrolls it so that v(k) is a register).
template <int LOOP, typename Get>
__device__ __forceinline__ void pixel_stats(Get v, int N, bool has_y, float y, float s, float* mean_out, float* spread_out,
                                            PixelAcc& acc, unsigned* hist) {
  double sum = 0.0;
#pragma unroll(LOOP <= 8 ? LOOP : 1)
  for (int k = 0; k < LOOP; ++k)
    if (k < N) sum += (double)v(k);
  const double mean = sum / N;
  double ss = 0.0, pw = 0.0, ae = 0.0;
  int below = 0;
#pragma unroll(LOOP <= 8 ? LOOP : 1)
  for (int k = 0; k < LOOP; ++k) {
    if (k < N) {
      const double x = (double)v(k);
      ss += (x - mean) * (x - mean);
      pw += (double)(2 * k - N + 1) * x;        // sorted order: sum_i sum_j |x_i - x_j| = 2 sum_k (2k - N + 1) x_(k)
      if (has_y) {
        ae += fabs(x - (double)y);
        below += v(k) < y ? 1 : 0;
      }
    }
  }
  const double var = ss / (N - 1);
  if (mean_out) *mean_out = (float)mean;
  if (spread_out) *spread_out = (float)sqrt(var);
  const double sd = (double)s;
  acc.q[3] += sd * sd * var;
  if (has_y) {
    const double d = mean - (double)y;
    acc.q[0] += sd * ae / N;
    acc.q[1] += sd * 2.0 * pw;
    acc.q[2] += sd * sd * d * d;
    acc.q[4] += sd * d;
    atomicAdd(hist + below, 1u);
  }
}

template <int BLOCK>
__device__ __forceinline__ void flush(PixelAcc& acc, const unsigned* hist, int N, bool has_y, int plane, double* gacc,
                                      unsigned long long* ghist) {
  __shared__ double red[BLOCK / 32][kEnsK];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < kEnsK; ++k) {
    double v = acc.q[k];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (lane == 0) red[warp][k] = v;
  }
  __syncthreads();
  if (threadIdx.x < kEnsK && (has_y || threadIdx.x == 3)) {
    double v = 0.0;
    for (int w = 0; w < BLOCK / 32; ++w) v += red[w][threadIdx.x];
    atomicAdd(gacc + (int64_t)plane * kEnsK + threadIdx.x, v);
  }
  if (has_y && ghist)
    for (int b = threadIdx.x; b <= N; b += BLOCK)
      if (hist[b]) atomicAdd(ghist + (int64_t)plane * (N + 1) + b, (unsigned long long)hist[b]);
}

// N <= NP <= 8: the members of a pixel in registers, padded with +inf and sorted by a bitonic network (constant indices).
template <int NP>
__global__ void __launch_bounds__(256) ens_stats_reg_kernel(const float* __restrict__ ens, int N, int64_t mstride,
                                                            const float* __restrict__ target, int64_t hw, const float* __restrict__ scale,
                                                            float* __restrict__ mean, float* __restrict__ spread, double* __restrict__ acc,
                                                            unsigned long long* __restrict__ rank_hist) {
  constexpr int BLOCK = 256;
  __shared__ unsigned hist[NP + 1];
  const int plane = blockIdx.y;
  for (int b = threadIdx.x; b <= N; b += BLOCK) hist[b] = 0u;
  __syncthreads();
  const float s = scale ? scale[plane] : 1.f;
  const int64_t base = (int64_t)plane * hw;
  PixelAcc pa;
  pa.zero();
  for (int64_t j = (int64_t)blockIdx.x * BLOCK + threadIdx.x; j < hw; j += (int64_t)gridDim.x * BLOCK) {
    float v[NP];
#pragma unroll
    for (int k = 0; k < NP; ++k) v[k] = k < N ? __ldg(ens + k * mstride + base + j) : __int_as_float(0x7f800000);
#pragma unroll
    for (int size = 2; size <= NP; size <<= 1)
#pragma unroll
      for (int stride = size >> 1; stride > 0; stride >>= 1)
#pragma unroll
        for (int k = 0; k < NP; ++k) {
          const int l = k ^ stride;
          if (l > k) {
            if ((k & size) == 0) cswap(v[k], v[l]);
            else cswap(v[l], v[k]);
          }
        }
    const float y = target ? target[base + j] : 0.f;
    // only v[k < N] is read: the network leaves the +inf padding at the end
    pixel_stats<NP>([&](int k) { return v[k]; }, N, target != nullptr, y, s, mean ? mean + base + j : nullptr, spread ? spread + base + j : nullptr, pa, hist);
  }
  __syncthreads();
  flush<BLOCK>(pa, hist, N, target != nullptr, plane, acc, rank_hist);
}

// 8 < N <= 256: each thread sorts its pixel's column s[k * BLOCK + tid], k < NP (power of two, +inf padded), in shared memory.
constexpr int kEnsSmemBlock = 64;
__global__ void __launch_bounds__(kEnsSmemBlock) ens_stats_smem_kernel(const float* __restrict__ ens, int N, int NP, int64_t mstride,
                                                                        const float* __restrict__ target, int64_t hw,
                                                                        const float* __restrict__ scale, float* __restrict__ mean,
                                                                        float* __restrict__ spread, double* __restrict__ acc,
                                                                        unsigned long long* __restrict__ rank_hist) {
  constexpr int BLOCK = kEnsSmemBlock;
  extern __shared__ float col[];
  __shared__ unsigned hist[257];
  const int plane = blockIdx.y, tid = threadIdx.x;
  for (int b = tid; b <= N; b += BLOCK) hist[b] = 0u;
  __syncthreads();
  const float s = scale ? scale[plane] : 1.f;
  const int64_t base = (int64_t)plane * hw;
  float* c = col + tid;
  PixelAcc pa;
  pa.zero();
  for (int64_t j = (int64_t)blockIdx.x * BLOCK + tid; j < hw; j += (int64_t)gridDim.x * BLOCK) {
    for (int k = 0; k < NP; ++k) c[k * BLOCK] = k < N ? __ldg(ens + k * mstride + base + j) : __int_as_float(0x7f800000);
    for (int size = 2; size <= NP; size <<= 1)
      for (int stride = size >> 1; stride > 0; stride >>= 1)
        for (int k = 0; k < NP; ++k) {
          const int l = k ^ stride;
          if (l > k) {
            float a = c[k * BLOCK], b = c[l * BLOCK];
            const bool up = (k & size) == 0;
            const float lo = fminf(a, b), hi = fmaxf(a, b);
            c[k * BLOCK] = up ? lo : hi;
            c[l * BLOCK] = up ? hi : lo;
          }
        }
    const float y = target ? target[base + j] : 0.f;
    pixel_stats<256>([&](int k) { return c[k * BLOCK]; }, N, target != nullptr, y, s, mean ? mean + base + j : nullptr,
                spread ? spread + base + j : nullptr, pa, hist);
  }
  __syncthreads();
  flush<BLOCK>(pa, hist, N, target != nullptr, plane, acc, rank_hist);
}

}  // namespace wsr

using namespace wsr;

extern "C" int wsr_ensemble_stats(const float* ens, int N, int64_t member_stride, const float* target, int planes, int64_t hw,
                                  const float* scale, float* mean, float* spread, double* acc, unsigned long long* rank_hist,
                                  void* stream) {
  WSR_REQUIRE(ens && acc && planes > 0 && hw > 0, WSR_E_INVALID, "ensemble_stats: bad argument");
  WSR_REQUIRE(N >= 2 && N <= 256, WSR_E_UNSUPPORTED, "ensemble_stats: N=%d outside 2..256", N);
  WSR_REQUIRE(member_stride >= (int64_t)planes * hw, WSR_E_INVALID, "ensemble_stats: member_stride %lld < planes * hw", (long long)member_stride);
  WSR_REQUIRE(planes <= 65535, WSR_E_UNSUPPORTED, "ensemble_stats: planes=%d > 65535", planes);
  cudaStream_t st = (cudaStream_t)stream;
  int np = 2;
  while (np < N) np <<= 1;
  // enough blocks per plane for ~8 resident blocks per SM over all planes, never more than the plane has pixels
  auto grid_x = [&](int block) {
    int64_t want = ((int64_t)148 * 8 + planes - 1) / planes;
    int64_t cap = (hw + block - 1) / block;
    return (unsigned)(want < cap ? (want < 1 ? 1 : want) : cap);
  };
  if (np <= 8) {
    dim3 grid(grid_x(256), planes);
    switch (np) {
      case 2: ens_stats_reg_kernel<2><<<grid, 256, 0, st>>>(ens, N, member_stride, target, hw, scale, mean, spread, acc, rank_hist); break;
      case 4: ens_stats_reg_kernel<4><<<grid, 256, 0, st>>>(ens, N, member_stride, target, hw, scale, mean, spread, acc, rank_hist); break;
      default: ens_stats_reg_kernel<8><<<grid, 256, 0, st>>>(ens, N, member_stride, target, hw, scale, mean, spread, acc, rank_hist); break;
    }
    WSR_LAUNCH_OK();
    return WSR_OK;
  }
  const size_t smem = (size_t)np * kEnsSmemBlock * sizeof(float);
  static size_t attr = 0;
  if (smem > attr) {
    WSR_CUDA_OK(cudaFuncSetAttribute(ens_stats_smem_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr = smem;
  }
  dim3 grid(grid_x(kEnsSmemBlock), planes);
  ens_stats_smem_kernel<<<grid, kEnsSmemBlock, smem, st>>>(ens, N, np, member_stride, target, hw, scale, mean, spread, acc, rank_hist);
  WSR_LAUNCH_OK();
  return WSR_OK;
}
