// backward.cu -- backward-pass kernels of the training step (reference: models/diffusion_models/model.py:61-69,
// `l_pix.backward()` through resdiff/unet.py:121-177): weight gradients of the tap-table convolutions, GroupNorm(+act,
// +dropout) backward, softmax backward, the noise-level embedding backward, FD_Info_Spliter gate backward, and Adam.
//
// Data gradients (dgrad) of the convolutions are NOT here: the gradient of a convolution w.r.t. its input is again a
// tap-table convolution (flipped / transposed weights), so it runs on the forward kernels (wsr_conv_tc /
// wsr_conv_taps_*).
#include "common.cuh"
#include "philox.cuh"

namespace wsr {

// ------------------------------------------------------------------------------------------------------------------
// weight gradient, SIMT fp32-accumulate:  dw[wtap][co][ci] += sum_{n, g} dy[n, g*out_mul + out_p, co] * X[n, in(g, tap), ci]
// GEMM view per tap: M = Cout, N = Cin, K = pixels.  grid = (co tiles, ci tiles, ntaps * splits); each block reduces a
// contiguous K range and adds its partial tile with fp32 atomics.
// ------------------------------------------------------------------------------------------------------------------
struct WgradParams {
  WsrWgradDesc d;
  WsrTapTable t;
  int splits;
  int64_t K;            // N * GH * GW
};

template <typename TX, typename TY>
__global__ void __launch_bounds__(256) conv_wgrad_simt_kernel(const WgradParams p) {
  constexpr int BM = 64, BN = 64, BK = 16;
  __shared__ float As[BK][BM + 4];   // dy:  [k][co]
  __shared__ float Bs[BK][BN + 4];   // x:   [k][ci]
  const WsrWgradDesc& d = p.d;
  const WsrTapTable& t = p.t;
  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;
  const int co0 = blockIdx.x * BM, ci0 = blockIdx.y * BN;
  const int tap = blockIdx.z / p.splits, split = blockIdx.z % p.splits;
  const int64_t kper = (p.K + p.splits - 1) / p.splits;
  const int64_t kbeg = (int64_t)split * kper;
  const int64_t kend = kbeg + kper < p.K ? kbeg + kper : p.K;
  const int in_stride = t.in_sub;
  const int dyt = t.in_sub * t.dy[tap] + t.py[tap], dxt = t.in_sub * t.dx[tap] + t.px[tap];
  const int UH = d.H * d.up, UW = d.W * d.up;
  const bool do_bias = d.dbias != nullptr && blockIdx.y == 0 && tap == 0;

  // loader mapping: thread -> (k row = tid / 16, 4 channels at (tid % 16) * 4)
  const int lk = tid >> 4, lc = (tid & 15) * 4;
  const TX* x = (const TX*)d.x;
  const TY* dy = (const TY*)d.dy;
  float acc[4][4];
  float bsum[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

  for (int64_t k0 = kbeg; k0 < kend; k0 += BK) {
    const int64_t k = k0 + lk;
    const TY* yp = nullptr;
    const TX* xp = nullptr;
    if (k < kend) {
      const int img = (int)(k / ((int64_t)t.GH * t.GW));
      const int r = (int)(k - (int64_t)img * t.GH * t.GW);
      const int gy = r / t.GW, gx = r - gy * t.GW;
      const int oy = gy * t.out_mul + t.out_py, ox = gx * t.out_mul + t.out_px;
      yp = dy + ((int64_t)(img * t.OH + oy) * t.OW + ox) * d.dy_ld;
      const int uy = gy * in_stride + dyt, ux = gx * in_stride + dxt;
      if (uy >= 0 && uy < UH && ux >= 0 && ux < UW) xp = x + ((int64_t)(img * d.H + uy / d.up) * d.W + ux / d.up) * d.x_ld;
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int co = co0 + lc + j, ci = ci0 + lc + j;
      As[lk][lc + j] = (yp && co < d.Cout) ? ldf<TY>(yp + co) : 0.f;
      Bs[lk][lc + j] = (xp && ci < d.Cin) ? ldf<TX>(xp + ci) : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < BK; ++kk) {
      float a[4], b[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) a[i] = As[kk][ty * 4 + i];
#pragma unroll
      for (int j = 0; j < 4; ++j) b[j] = Bs[kk][tx * 4 + j];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
      if (do_bias && tx == 0) {
#pragma unroll
        for (int i = 0; i < 4; ++i) bsum[i] += a[i];
      }
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int co = co0 + ty * 4 + i;
    if (co >= d.Cout) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int ci = ci0 + tx * 4 + j;
      if (ci >= d.Cin) continue;
      atomicAdd(d.dw + (int64_t)t.wtap[tap] * d.dw_stap + (int64_t)co * d.dw_sco + (int64_t)ci * d.dw_sci, acc[i][j]);
    }
    if (do_bias && tx == 0) atomicAdd(d.dbias + co, bsum[i]);
  }
}

// ------------------------------------------------------------------------------------------------------------------
// GroupNorm (+ activation, + dropout) backward.
//   forward:  xh = (x - mean_g) * rstd_g ;  z = xh * gamma_c + beta_c ;  a = act(z) * drop
//   given da: dz = da * drop * act'(z)
//   pass 1 (reduce):  red[n][c] = (sum_p dz, sum_p dz * xh)
//   pass 2 (apply):   dx (+)= rstd * (dz * gamma - A_g / m - xh * B_g / m),  A_g = sum_{c in g} gamma_c red0, B_g = ... red1
//                     block (0, 0) also emits dgamma += sum_n red1, dbeta += sum_n red0 and (optionally) the per-image
//                     column sums of dx, which are known in closed form from red and the forward statistics.
// ------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ float act_grad(float z, int act) {
  switch (act) {
    case WSR_ACT_SWISH: { float s = 1.f / (1.f + expf(-z)); return s * (1.f + z * (1.f - s)); }
    case WSR_ACT_RELU: return z > 0.f ? 1.f : 0.f;
    case WSR_ACT_LRELU02: return z > 0.f ? 1.f : 0.2f;
    case WSR_ACT_MISH: {
      float sp = z > 20.f ? z : log1pf(expf(z));
      float th = tanhf(sp);
      float sg = 1.f / (1.f + expf(-z));
      return th + z * sg * (1.f - th * th);
    }
    default: return 1.f;
  }
}

// group statistics of image n -> per-channel (mean, rstd) pairs in shared memory
// Group-first: ONE thread per group sums the group's per-channel statistics and takes the (double precision) division and
// reciprocal square root, then every channel copies its group's pair (the per-channel version repeated that work cpg times in
// every block).  Must be called by all threads of the block; ends with a barrier.
// Measured: no change of the small-tensor launch time (22 us at B = 4, 8x16x512).  ncu on that launch: 32 blocks, ~3500
// straight-line SASS instructions per warp at ~14 cycles each (issue slots 14 % busy, DRAM 0.9 %): the launch is one long
// dependent chain per warp (statistics loads -> moments -> 4 pixels x 8 channels with the activation gradient -> shared and
// global double atomics), not a throughput problem.
__device__ __forceinline__ void gn_channel_moments(const double* stats, int stats_ld, int n, int C, int groups, int HW, float eps,
                                                   float* mean_s, float* rstd_s) {
  const int cpg = C / groups;
  for (int g = threadIdx.x; g < groups; g += blockDim.x) {
    const int g0 = g * cpg;
    double a = 0.0, b = 0.0;
    for (int j = 0; j < cpg; ++j) { a += stats[(int64_t)n * stats_ld + (g0 + j) * 2]; b += stats[(int64_t)n * stats_ld + (g0 + j) * 2 + 1]; }
    const double cnt = (double)cpg * HW;
    const double mean = a / cnt;
    double var = b / cnt - mean * mean;
    if (var < 0.0) var = 0.0;
    mean_s[g0] = (float)mean;                                  // parked in the group's first channel slot
    rstd_s[g0] = (float)(1.0 / sqrt(var + (double)eps));
  }
  __syncthreads();
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    const int g0 = (c / cpg) * cpg;
    if (c != g0) { mean_s[c] = mean_s[g0]; rstd_s[c] = rstd_s[g0]; }
  }
  __syncthreads();
}

// ga[c] = sum_{j in group(c)} gamma[j] * red[n][2j] / (cpg * HW), gb[c] likewise with red[n][2j + 1]: same group-first scheme
__device__ __forceinline__ void gn_group_sums(const float* gamma, const double* red, int red_ld, int n, int C, int groups, int HW,
                                              float* ga, float* gb) {
  const int cpg = C / groups;
  for (int g = threadIdx.x; g < groups; g += blockDim.x) {
    const int g0 = g * cpg;
    double A = 0.0, Bq = 0.0;
    for (int j = 0; j < cpg; ++j) {
      A += (double)gamma[g0 + j] * red[(int64_t)n * red_ld + 2 * (g0 + j)];
      Bq += (double)gamma[g0 + j] * red[(int64_t)n * red_ld + 2 * (g0 + j) + 1];
    }
    const double m = (double)cpg * HW;
    ga[g0] = (float)(A / m);
    gb[g0] = (float)(Bq / m);
  }
  __syncthreads();
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    const int g0 = (c / cpg) * cpg;
    if (c != g0) { ga[c] = ga[g0]; gb[c] = gb[g0]; }
  }
}

struct GnBwdArgs {
  const void* x; int HW, C, x_ld;
  const double* stats; int stats_ld;
  const float* gamma; const float* beta; int groups; float eps; int act;
  const void* da; int da_ld;
  float drop_p; uint64_t drop_seed; uint32_t drop_tag;
  double* red; int red_ld;
  void* dx; int dx_ld;
  float* dgamma; float* dbeta; float* colsum; int colsum_ld; int N;
  int chunk;
};

template <typename T>
__global__ void __launch_bounds__(256) gn_bwd_reduce_kernel(const GnBwdArgs a) {
  extern __shared__ float sm[];   // mean[C], rstd[C]
  float* mean_s = sm;
  float* rstd_s = sm + a.C;
  const int n = blockIdx.y;
  gn_channel_moments(a.stats, a.stats_ld, n, a.C, a.groups, a.HW, a.eps, mean_s, rstd_s);
  __syncthreads();
  const int p0 = blockIdx.x * a.chunk, p1 = min(a.HW, p0 + a.chunk);
  const T* x = (const T*)a.x + (int64_t)n * a.HW * a.x_ld;
  const T* da = (const T*)a.da + (int64_t)n * a.HW * a.da_ld;
  // thread -> channel c (strided by blockDim), loops over the pixel chunk: coalesced over channels
  for (int c = threadIdx.x; c < a.C; c += blockDim.x) {
    const float mu = mean_s[c], rs = rstd_s[c], g = a.gamma[c], b = a.beta[c];
    float s0 = 0.f, s1 = 0.f;
    for (int p = p0; p < p1; ++p) {
      const float xh = (ldf<T>(x + (int64_t)p * a.x_ld + c) - mu) * rs;
      float dz = ldf<T>(da + (int64_t)p * a.da_ld + c) * act_grad(fmaf(xh, g, b), a.act);
      if (a.drop_p > 0.f) {
        float m[1];
        dropout_scale<1>(a.drop_seed, a.drop_tag, ((uint64_t)n * a.HW + (uint64_t)p) * a.C + (uint64_t)c, a.drop_p, m);
        dz *= m[0];
      }
      s0 += dz;
      s1 = fmaf(dz, xh, s1);
    }
    atomicAdd(&a.red[(int64_t)n * a.red_ld + 2 * c], (double)s0);
    atomicAdd(&a.red[(int64_t)n * a.red_ld + 2 * c + 1], (double)s1);
  }
}

template <typename T>
__global__ void __launch_bounds__(256) gn_bwd_apply_kernel(const GnBwdArgs a, int accumulate) {
  extern __shared__ float sm[];   // mean[C], rstd[C], ga[C] (A_g / m per channel), gb[C] (B_g / m per channel)
  float* mean_s = sm;
  float* rstd_s = sm + a.C;
  float* ga = sm + 2 * a.C;
  float* gb = sm + 3 * a.C;
  const int n = blockIdx.y;
  const int cpg = a.C / a.groups;
  gn_channel_moments(a.stats, a.stats_ld, n, a.C, a.groups, a.HW, a.eps, mean_s, rstd_s);
  gn_group_sums(a.gamma, a.red, a.red_ld, n, a.C, a.groups, a.HW, ga, gb);
  __syncthreads();
  const int p0 = blockIdx.x * a.chunk, p1 = min(a.HW, p0 + a.chunk);
  const T* x = (const T*)a.x + (int64_t)n * a.HW * a.x_ld;
  const T* da = (const T*)a.da + (int64_t)n * a.HW * a.da_ld;
  T* dx = (T*)a.dx + (int64_t)n * a.HW * a.dx_ld;
  for (int c = threadIdx.x; c < a.C; c += blockDim.x) {
    const float mu = mean_s[c], rs = rstd_s[c], g = a.gamma[c], b = a.beta[c], A = ga[c], Bq = gb[c];
    for (int p = p0; p < p1; ++p) {
      const float xh = (ldf<T>(x + (int64_t)p * a.x_ld + c) - mu) * rs;
      float dz = ldf<T>(da + (int64_t)p * a.da_ld + c) * act_grad(fmaf(xh, g, b), a.act);
      if (a.drop_p > 0.f) {
        float m[1];
        dropout_scale<1>(a.drop_seed, a.drop_tag, ((uint64_t)n * a.HW + (uint64_t)p) * a.C + (uint64_t)c, a.drop_p, m);
        dz *= m[0];
      }
      float v = rs * (dz * g - A - xh * Bq);
      T* o = dx + (int64_t)p * a.dx_ld + c;
      if (accumulate) v += ldf<T>(o);
      stf<T>(o, v);
    }
  }
  // parameter gradients and closed-form column sums: one block per image handles its own column sums, block (0,0) the
  // batch-summed parameter gradients
  if (blockIdx.x == 0) {
    if (a.colsum) {
      // sum_p dx[n,p,c] = rstd * (gamma_c * red0 - HW * A_g/m - (sum_p xh) * B_g/m),  sum_p xh = (sum_x - HW*mean) * rstd
      for (int c = threadIdx.x; c < a.C; c += blockDim.x) {
        const double sx = a.stats[(int64_t)n * a.stats_ld + 2 * c];
        const double sxh = (sx - (double)a.HW * mean_s[c]) * rstd_s[c];
        const double v = (double)rstd_s[c] * ((double)a.gamma[c] * a.red[(int64_t)n * a.red_ld + 2 * c] - (double)a.HW * ga[c] - sxh * gb[c]);
        a.colsum[(int64_t)n * a.colsum_ld + c] = (float)v;
      }
    }
    if (n == 0 && a.dgamma) {
      for (int c = threadIdx.x; c < a.C; c += blockDim.x) {
        double s0 = 0.0, s1 = 0.0;
        for (int i = 0; i < a.N; ++i) { s0 += a.red[(int64_t)i * a.red_ld + 2 * c]; s1 += a.red[(int64_t)i * a.red_ld + 2 * c + 1]; }
        a.dgamma[c] += (float)s1;
        a.dbeta[c] += (float)s0;
      }
    }
  }
}

// Vectorised versions (16-byte accesses: 8 bf16 / 4 fp32 channels per thread; thread t owns channel vector t % CV and pixel
// lane t / CV, like gn_apply_kernel).  The scalar kernels above remain for pitches / widths that are not vector-aligned.
template <typename T, int VEC>
__device__ __forceinline__ void gn_bwd_dz(const GnBwdArgs& a, int n, int p, int cv, const T* x, const T* da, const float (&mu)[VEC],
                                          const float (&rs)[VEC], const float (&g)[VEC], const float (&b)[VEC], float (&xh)[VEC],
                                          float (&dz)[VEC]) {
  float xv[VEC], dv[VEC];
  VecLoad<T, VEC>::ld(x + (int64_t)p * a.x_ld, xv);
  VecLoad<T, VEC>::ld(da + (int64_t)p * a.da_ld, dv);
#pragma unroll
  for (int i = 0; i < VEC; ++i) {
    xh[i] = (xv[i] - mu[i]) * rs[i];
    dz[i] = dv[i] * act_grad(fmaf(xh[i], g[i], b[i]), a.act);
  }
  if (a.drop_p > 0.f) {
    float m[VEC];
    dropout_scale<VEC>(a.drop_seed, a.drop_tag, ((uint64_t)n * a.HW + (uint64_t)p) * a.C + (uint64_t)cv * VEC, a.drop_p, m);
#pragma unroll
    for (int i = 0; i < VEC; ++i) dz[i] *= m[i];
  }
}

template <typename T, int VEC>
__global__ void __launch_bounds__(1024) gn_bwd_reduce_vec_kernel(const GnBwdArgs a, int CV, int PL) {
  extern __shared__ float sm[];   // mean[C], rstd[C], acc[2C]
  float* mean_s = sm;
  float* rstd_s = sm + a.C;
  float* acc = sm + 2 * a.C;
  const int n = blockIdx.y;
  gn_channel_moments(a.stats, a.stats_ld, n, a.C, a.groups, a.HW, a.eps, mean_s, rstd_s);
  for (int c = threadIdx.x; c < 2 * a.C; c += blockDim.x) acc[c] = 0.f;
  __syncthreads();
  const int cv = threadIdx.x % CV, pl = threadIdx.x / CV;
  const int p0 = blockIdx.x * a.chunk, p1 = min(a.HW, p0 + a.chunk);
  const T* x = (const T*)a.x + (int64_t)n * a.HW * a.x_ld + cv * VEC;
  const T* da = (const T*)a.da + (int64_t)n * a.HW * a.da_ld + cv * VEC;
  float mu[VEC], rs[VEC], g[VEC], b[VEC], s0[VEC], s1[VEC];
#pragma unroll
  for (int i = 0; i < VEC; ++i) {
    const int c = cv * VEC + i;
    mu[i] = mean_s[c]; rs[i] = rstd_s[c]; g[i] = a.gamma[c]; b[i] = a.beta[c]; s0[i] = 0.f; s1[i] = 0.f;
  }
  for (int p = p0 + pl; p < p1; p += PL) {
    float xh[VEC], dz[VEC];
    gn_bwd_dz<T, VEC>(a, n, p, cv, x, da, mu, rs, g, b, xh, dz);
#pragma unroll
    for (int i = 0; i < VEC; ++i) { s0[i] += dz[i]; s1[i] = fmaf(dz[i], xh[i], s1[i]); }
  }
#pragma unroll
  for (int i = 0; i < VEC; ++i) {
    atomicAdd(&acc[2 * (cv * VEC + i)], s0[i]);
    atomicAdd(&acc[2 * (cv * VEC + i) + 1], s1[i]);
  }
  __syncthreads();
  for (int c = threadIdx.x; c < 2 * a.C; c += blockDim.x) atomicAdd(&a.red[(int64_t)n * a.red_ld + c], (double)acc[c]);
}

template <typename T, int VEC>
__global__ void __launch_bounds__(1024) gn_bwd_apply_vec_kernel(const GnBwdArgs a, int accumulate, int CV, int PL) {
  extern __shared__ float sm[];   // mean[C], rstd[C], ga[C], gb[C]
  float* mean_s = sm;
  float* rstd_s = sm + a.C;
  float* ga = sm + 2 * a.C;
  float* gb = sm + 3 * a.C;
  const int n = blockIdx.y;
  const int cpg = a.C / a.groups;
  gn_channel_moments(a.stats, a.stats_ld, n, a.C, a.groups, a.HW, a.eps, mean_s, rstd_s);
  gn_group_sums(a.gamma, a.red, a.red_ld, n, a.C, a.groups, a.HW, ga, gb);
  __syncthreads();
  const int cv = threadIdx.x % CV, pl = threadIdx.x / CV;
  const int p0 = blockIdx.x * a.chunk, p1 = min(a.HW, p0 + a.chunk);
  const T* x = (const T*)a.x + (int64_t)n * a.HW * a.x_ld + cv * VEC;
  const T* da = (const T*)a.da + (int64_t)n * a.HW * a.da_ld + cv * VEC;
  T* dx = (T*)a.dx + (int64_t)n * a.HW * a.dx_ld + cv * VEC;
  float mu[VEC], rs[VEC], g[VEC], b[VEC], A[VEC], Bq[VEC];
#pragma unroll
  for (int i = 0; i < VEC; ++i) {
    const int c = cv * VEC + i;
    mu[i] = mean_s[c]; rs[i] = rstd_s[c]; g[i] = a.gamma[c]; b[i] = a.beta[c]; A[i] = ga[c]; Bq[i] = gb[c];
  }
  for (int p = p0 + pl; p < p1; p += PL) {
    float xh[VEC], dz[VEC], v[VEC];
    gn_bwd_dz<T, VEC>(a, n, p, cv, x, da, mu, rs, g, b, xh, dz);
#pragma unroll
    for (int i = 0; i < VEC; ++i) v[i] = rs[i] * (dz[i] * g[i] - A[i] - xh[i] * Bq[i]);
    T* o = dx + (int64_t)p * a.dx_ld;
    if (accumulate) {
      float old[VEC];
      VecLoad<T, VEC>::ld(o, old);
#pragma unroll
      for (int i = 0; i < VEC; ++i) v[i] += old[i];
    }
    VecLoad<T, VEC>::st(o, v);
  }
  if (blockIdx.x == 0) {
    if (a.colsum) {
      for (int c = threadIdx.x; c < a.C; c += blockDim.x) {
        const double sx = a.stats[(int64_t)n * a.stats_ld + 2 * c];
        const double sxh = (sx - (double)a.HW * mean_s[c]) * rstd_s[c];
        const double v = (double)rstd_s[c] * ((double)a.gamma[c] * a.red[(int64_t)n * a.red_ld + 2 * c] - (double)a.HW * ga[c] - sxh * gb[c]);
        a.colsum[(int64_t)n * a.colsum_ld + c] = (float)v;
      }
    }
    if (n == 0 && a.dgamma) {
      for (int c = threadIdx.x; c < a.C; c += blockDim.x) {
        double s0 = 0.0, s1 = 0.0;
        for (int i = 0; i < a.N; ++i) { s0 += a.red[(int64_t)i * a.red_ld + 2 * c]; s1 += a.red[(int64_t)i * a.red_ld + 2 * c + 1]; }
        a.dgamma[c] += (float)s1;
        a.dbeta[c] += (float)s0;
      }
    }
  }
}

// vector width usable for (x, da[, dx]): 8 (bf16) / 4 (fp32) when widths, pitches and addresses allow 16-byte accesses
static int gn_bwd_vec(int dt, int C, int x_ld, int da_ld, int dx_ld, const void* x, const void* da, const void* dx) {
  const int want = dt == WSR_BF16 ? 8 : 4;
  const bool ok = C % want == 0 && x_ld % want == 0 && da_ld % want == 0 && dx_ld % want == 0 && (((uintptr_t)x | (uintptr_t)da | (uintptr_t)dx) & 15) == 0 &&
                  C / want <= 1024;
  return ok ? want : 1;
}

// ------------------------------------------------------------------------------------------------------------------
// softmax backward: ds[r][c] = scale * p[r][c] * (dp[r][c] - sum_c' dp[r][c'] p[r][c'])
// ------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ float warp_sum_b(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

__global__ void __launch_bounds__(128) softmax_bwd_rows_kernel(const void* p, int pdt, const void* dp, int dpdt, int cols,
                                                              int64_t ld, float scale, void* ds, int dsdt) {
  __shared__ float red[4];
  const int64_t r = blockIdx.x;
  float acc = 0.f;
  for (int c = threadIdx.x; c < cols; c += 128) acc = fmaf(ld_dt(p, r * ld + c, pdt), ld_dt(dp, r * ld + c, dpdt), acc);
  acc = warp_sum_b(acc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  const float dot = red[0] + red[1] + red[2] + red[3];
  for (int c = threadIdx.x; c < cols; c += 128) {
    const float pv = ld_dt(p, r * ld + c, pdt);
    st_dt(ds, r * ld + c, dsdt, scale * pv * (ld_dt(dp, r * ld + c, dpdt) - dot));
  }
}

// ------------------------------------------------------------------------------------------------------------------
// noise-level embedding backward (PositionalEncoding has no parameters; the level itself needs no gradient)
//   temb = W2 act(W1 enc + b1) + b2   ->  dW2, db2, dW1, db1 (+=, atomics over the R rows)
// ------------------------------------------------------------------------------------------------------------------
__global__ void noise_embed_bwd_kernel(const float* __restrict__ level, int inner, const float* __restrict__ w1,
                                       const float* __restrict__ b1, const float* __restrict__ w2, int act,
                                       const float* __restrict__ dtemb, float* dw1, float* db1, float* dw2, float* db2) {
  extern __shared__ float sm[];   // enc[inner], pre[4*inner], hid[4*inner], dpre[4*inner], dt[inner]
  float* enc = sm;
  float* pre = enc + inner;
  float* hid = pre + 4 * inner;
  float* dpre = hid + 4 * inner;
  float* dt = dpre + 4 * inner;
  const int r = blockIdx.x;
  const float lv = level[r];
  const int half = inner / 2;
  for (int k = threadIdx.x; k < half; k += blockDim.x) {
    float step = (float)k / (float)half;
    float arg = lv * expf(-logf(1e4f) * step);
    enc[k] = sinf(arg);
    enc[half + k] = cosf(arg);
  }
  for (int o = threadIdx.x; o < inner; o += blockDim.x) dt[o] = dtemb[(int64_t)r * inner + o];
  __syncthreads();
  for (int o = threadIdx.x; o < 4 * inner; o += blockDim.x) {
    float a = b1[o];
    for (int k = 0; k < inner; ++k) a = fmaf(w1[(int64_t)o * inner + k], enc[k], a);
    pre[o] = a;
    hid[o] = apply_act(a, act);
  }
  __syncthreads();
  // dW2[o][k] += dt[o] * hid[k]; db2[o] += dt[o]; dhid[k] = sum_o dt[o] * W2[o][k]
  for (int i = threadIdx.x; i < inner * 4 * inner; i += blockDim.x) {
    const int o = i / (4 * inner), k = i - o * 4 * inner;
    atomicAdd(dw2 + i, dt[o] * hid[k]);
  }
  for (int o = threadIdx.x; o < inner; o += blockDim.x) atomicAdd(db2 + o, dt[o]);
  for (int k = threadIdx.x; k < 4 * inner; k += blockDim.x) {
    float a = 0.f;
    for (int o = 0; o < inner; ++o) a = fmaf(dt[o], w2[(int64_t)o * 4 * inner + k], a);
    dpre[k] = a * act_grad(pre[k], act);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 4 * inner * inner; i += blockDim.x) {
    const int o = i / inner, k = i - o * inner;
    atomicAdd(dw1 + i, dpre[o] * enc[k]);
  }
  for (int o = threadIdx.x; o < 4 * inner; o += blockDim.x) atomicAdd(db1 + o, dpre[o]);
}

// y[r][o] = b[o] + sum_k w[o][k] x[r][k]  ->  dw[o][k] += sum_r dy[r][o] x[r][k]; db[o] += sum_r dy[r][o]
__global__ void linear_rows_bwd_w_kernel(const float* __restrict__ x, int R, int K, const float* __restrict__ dy, int P,
                                         float* dw, float* db) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;   // over P*K
  if (i >= (int64_t)P * K) return;
  const int o = (int)(i / K), k = (int)(i - (int64_t)o * K);
  float a = 0.f, bsum = 0.f;
  for (int r = 0; r < R; ++r) { const float g = dy[(int64_t)r * P + o]; a = fmaf(g, x[(int64_t)r * K + k], a); bsum += g; }
  dw[i] += a;
  if (k == 0 && db) db[o] += bsum;
}
// dx[r][k] = sum_o dy[r][o] w[o][k]
__global__ void linear_rows_bwd_x_kernel(const float* __restrict__ w, int K, const float* __restrict__ dy, int P, float* __restrict__ dx) {
  __shared__ float red[8];
  const int r = blockIdx.y, k = blockIdx.x;
  float a = 0.f;
  for (int o = threadIdx.x; o < P; o += blockDim.x) a = fmaf(dy[(int64_t)r * P + o], w[(int64_t)o * K + k], a);
  a = warp_sum_b(a);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = a;
  __syncthreads();
  if (threadIdx.x == 0) {
    float s = 0.f;
    for (int i = 0; i < (int)(blockDim.x >> 5); ++i) s += red[i];
    dx[(int64_t)r * K + k] = s;
  }
}

// ------------------------------------------------------------------------------------------------------------------
// FD_Info_Spliter gate backward (fd_info_spliter.py:43-47; forward = fd_gate_kernel + stem channel 2):
//   denoise_x[b,c,h,w] = x[b,c,h,w] * gate[b,c,w],  gate = ne[w] * (1 + se[c]),  se = sigmoid(fc2 relu(fc0 * mean_w ne))
//   in: dxin NHWC fp32/bf16 (channel 2C + c holds d denoise_x), x_t NCHW.  out: dne[b][w] (=), dfc0, dfc2 (+=)
// ------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) fd_gate_bwd_kernel(const void* dxin, int ddt, int d_ld, int ch0, const float* __restrict__ x,
                                                         const float* __restrict__ ne_rows, int ne_ld, int C, int H, int W,
                                                         const float* __restrict__ fc0, const float* __restrict__ fc2, int hidden,
                                                         float* __restrict__ dne, int dne_ld, float* dfc0, float* dfc2) {
  extern __shared__ float sm[];   // dgate[C*W], se[C], hid[hidden], a1[hidden], dse[C], scal[4]
  float* dgate = sm;
  float* se = dgate + C * W;
  float* hid = se + C;
  float* a1 = hid + hidden;
  float* dse = a1 + hidden;
  float* scal = dse + C;
  const int b = blockIdx.x;
  const float* ne = ne_rows + (int64_t)b * ne_ld;
  // dgate[c][w] = sum_h dxin[b,h,w,ch0+c] * x[b,c,h,w]
  for (int i = threadIdx.x; i < C * W; i += blockDim.x) {
    const int c = i / W, w = i - c * W;
    float a = 0.f;
    for (int h = 0; h < H; ++h)
      a = fmaf(ld_dt(dxin, ((int64_t)(b * H + h) * W + w) * d_ld + ch0 + c, ddt), x[((int64_t)(b * C + c) * H + h) * W + w], a);
    dgate[i] = a;
  }
  if (threadIdx.x == 0) {
    float m = 0.f;
    for (int w = 0; w < W; ++w) m += ne[w];
    m /= (float)W;
    for (int h = 0; h < hidden; ++h) {
      float a = 0.f;
      for (int c = 0; c < C; ++c) a = fmaf(fc0[h * C + c], m, a);
      a1[h] = a;
      hid[h] = a > 0.f ? a : 0.f;
    }
    for (int c = 0; c < C; ++c) {
      float a = 0.f;
      for (int h = 0; h < hidden; ++h) a = fmaf(fc2[c * hidden + h], hid[h], a);
      se[c] = 1.f / (1.f + expf(-a));
    }
    scal[0] = m;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    const float m = scal[0];
    for (int c = 0; c < C; ++c) {
      float a = 0.f;
      for (int w = 0; w < W; ++w) a = fmaf(dgate[c * W + w], ne[w], a);
      dse[c] = a * se[c] * (1.f - se[c]);       // d pre-sigmoid
    }
    float dm = 0.f;
    for (int h = 0; h < hidden; ++h) {
      float dh = 0.f;
      for (int c = 0; c < C; ++c) { dh = fmaf(dse[c], fc2[c * hidden + h], dh); atomicAdd(dfc2 + c * hidden + h, dse[c] * hid[h]); }
      const float da1 = a1[h] > 0.f ? dh : 0.f;
      float rowsum = 0.f;
      for (int c = 0; c < C; ++c) { atomicAdd(dfc0 + h * C + c, da1 * m); rowsum += fc0[h * C + c]; }
      dm = fmaf(da1, rowsum, dm);
    }
    scal[1] = dm / (float)W;
  }
  __syncthreads();
  for (int w = threadIdx.x; w < W; w += blockDim.x) {
    float a = scal[1];
    for (int c = 0; c < C; ++c) a = fmaf(dgate[c * W + w], 1.f + se[c], a);
    dne[(int64_t)b * dne_ld + w] = a;
  }
}

// ------------------------------------------------------------------------------------------------------------------
// Adam (torch.optim.Adam semantics, models/diffusion_models/model.py:43-44: lr, betas (0.9, 0.999), eps 1e-8, wd 0)
// With EMA the updated parameter, still in a register, also moves the exponential moving average:
// ema = ema * d + (1 - d) * p_new as three separately rounded fp32 operations (torch's expression with a Python-float d;
// __fmul_rn / __fadd_rn keep the compiler from contracting them into an FMA), or ema = p_new exactly when d == 0.
// ------------------------------------------------------------------------------------------------------------------
template <bool EMA>
__global__ void adam_step_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v,
                                 int64_t n, float lr, float b1, float b2, float omb1, float omb2, float eps, float wd, float bc1,
                                 float bc2_sqrt, float* __restrict__ ema, float ema_d, float ema_omd) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    float gi = g[i];
    const float pi = p[i];
    const float ei = EMA ? ema[i] : 0.f;             // issued with the other loads, not after the stores
    if (wd != 0.f) gi = fmaf(wd, pi, gi);
    const float mi = b1 * m[i] + omb1 * gi;          // 1 - beta rounded from double, as torch does
    const float vi = b2 * v[i] + omb2 * gi * gi;
    m[i] = mi; v[i] = vi;
    const float denom = sqrtf(vi) / bc2_sqrt + eps;
    const float pn = pi - (lr / bc1) * (mi / denom);
    p[i] = pn;
    if constexpr (EMA) ema[i] = ema_d == 0.f ? pn : __fadd_rn(__fmul_rn(ei, ema_d), __fmul_rn(ema_omd, pn));
  }
}

int validate_taps(const WsrTapTable* t);

}  // namespace wsr

using namespace wsr;

extern "C" int wsr_conv_wgrad_simt(const WsrWgradDesc* d, const WsrTapTable* t, void* stream) {
  WSR_REQUIRE(d && t, WSR_E_INVALID, "wgrad: null descriptor");
  WSR_REQUIRE(d->x && d->dy && d->dw, WSR_E_INVALID, "wgrad: null x/dy/dw");
  WSR_REQUIRE(valid_dtype(d->x_dtype) && valid_dtype(d->dy_dtype), WSR_E_INVALID, "wgrad: bad dtype");
  WSR_REQUIRE(d->N > 0 && d->H > 0 && d->W > 0 && d->Cin > 0 && d->Cout > 0 && d->x_ld >= d->Cin && d->dy_ld >= d->Cout,
              WSR_E_INVALID, "wgrad: bad shape");
  WSR_REQUIRE(d->up == 1 || d->up == 2, WSR_E_INVALID, "wgrad: up must be 1 or 2");
  int rc = validate_taps(t);
  if (rc) return rc;
  WgradParams p;
  p.d = *d; p.t = *t;
  p.K = (int64_t)d->N * t->GH * t->GW;
  const int tiles = ((d->Cout + 63) / 64) * ((d->Cin + 63) / 64) * t->ntaps;
  int splits = (592 + tiles - 1) / tiles;                     // ~4 blocks per SM
  const int64_t max_splits = (p.K + 255) / 256;
  if (splits > max_splits) splits = (int)max_splits;
  if (splits < 1) splits = 1;
  WSR_REQUIRE((int64_t)t->ntaps * splits <= 65535, WSR_E_UNSUPPORTED, "wgrad: grid z too large");
  p.splits = splits;
  dim3 grid((d->Cout + 63) / 64, (d->Cin + 63) / 64, t->ntaps * splits);
  cudaStream_t st = (cudaStream_t)stream;
  if (d->x_dtype == WSR_BF16 && d->dy_dtype == WSR_BF16) conv_wgrad_simt_kernel<__nv_bfloat16, __nv_bfloat16><<<grid, 256, 0, st>>>(p);
  else if (d->x_dtype == WSR_BF16) conv_wgrad_simt_kernel<__nv_bfloat16, float><<<grid, 256, 0, st>>>(p);
  else if (d->dy_dtype == WSR_BF16) conv_wgrad_simt_kernel<float, __nv_bfloat16><<<grid, 256, 0, st>>>(p);
  else conv_wgrad_simt_kernel<float, float><<<grid, 256, 0, st>>>(p);
  WSR_LAUNCH_OK();
  return WSR_OK;
}

static int gn_bwd_common(GnBwdArgs& a, const void* x, int x_dtype, int N, int HW, int C, int x_ld, const double* stats,
                         int stats_ld, const float* gamma, const float* beta, int groups, float eps, int act, const void* da,
                         int da_dtype, int da_ld, float drop_p, uint64_t drop_seed, uint32_t drop_tag, double* red, int red_ld) {
  WSR_REQUIRE(x && stats && gamma && beta && da && red, WSR_E_INVALID, "gn_bwd: null pointer");
  WSR_REQUIRE(valid_dtype(x_dtype) && da_dtype == x_dtype, WSR_E_UNSUPPORTED, "gn_bwd: da dtype must equal x dtype");
  WSR_REQUIRE(N > 0 && HW > 0 && C > 0 && x_ld >= C && da_ld >= C && stats_ld >= 2 * C && red_ld >= 2 * C, WSR_E_INVALID, "gn_bwd: bad shape");
  WSR_REQUIRE(groups > 0 && C % groups == 0, WSR_E_INVALID, "gn_bwd: C=%d not divisible by groups=%d", C, groups);
  WSR_REQUIRE(C <= 8192, WSR_E_UNSUPPORTED, "gn_bwd: C=%d too wide", C);
  WSR_REQUIRE(drop_p >= 0.f && drop_p < 1.f, WSR_E_INVALID, "gn_bwd: dropout p");
  a = GnBwdArgs{};
  a.x = x; a.HW = HW; a.C = C; a.x_ld = x_ld; a.stats = stats; a.stats_ld = stats_ld; a.gamma = gamma; a.beta = beta;
  a.groups = groups; a.eps = eps; a.act = act; a.da = da; a.da_ld = da_ld; a.drop_p = drop_p; a.drop_seed = drop_seed;
  a.drop_tag = drop_tag; a.red = red; a.red_ld = red_ld; a.N = N;
  // pixels per block: enough blocks to fill the machine, at least 8 pixels each
  int64_t want_blocks = 1184;       // measured at B = 4: 592 / 296 / 148 blocks change the step time by < 1 % either way
  int chunk = (int)(((int64_t)N * HW + want_blocks - 1) / want_blocks);
  if (chunk < 8) chunk = 8;
  if (chunk > HW) chunk = HW;
  a.chunk = chunk;
  return WSR_OK;
}

extern "C" int wsr_gn_bwd_reduce(const void* x, int x_dtype, int N, int HW, int C, int x_ld, const double* stats, int stats_ld,
                                 const float* gamma, const float* beta, int groups, float eps, int act, const void* da,
                                 int da_dtype, int da_ld, float drop_p, uint64_t drop_seed, uint32_t drop_tag, double* red,
                                 int red_ld, void* stream) {
  GnBwdArgs a;
  int rc = gn_bwd_common(a, x, x_dtype, N, HW, C, x_ld, stats, stats_ld, gamma, beta, groups, eps, act, da, da_dtype, da_ld, drop_p,
                         drop_seed, drop_tag, red, red_ld);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  const int vec = gn_bwd_vec(x_dtype, C, x_ld, da_ld, x_ld, x, da, x);
  if (vec > 1 && (size_t)4 * C * sizeof(float) <= 48 * 1024) {
    const int CV = C / vec, PL = CV >= 256 ? 1 : 256 / CV;
    if (a.chunk < 4 * PL) a.chunk = 4 * PL < HW ? 4 * PL : HW;
    dim3 grid((HW + a.chunk - 1) / a.chunk, N);
    size_t smem = (size_t)4 * C * sizeof(float);
    if (x_dtype == WSR_BF16) gn_bwd_reduce_vec_kernel<__nv_bfloat16, 8><<<grid, CV * PL, smem, st>>>(a, CV, PL);
    else gn_bwd_reduce_vec_kernel<float, 4><<<grid, CV * PL, smem, st>>>(a, CV, PL);
    WSR_LAUNCH_OK();
    return WSR_OK;
  }
  dim3 grid((HW + a.chunk - 1) / a.chunk, N);
  const int threads = C >= 256 ? 256 : ((C + 31) / 32) * 32;
  size_t smem = (size_t)2 * C * sizeof(float);
  if (x_dtype == WSR_BF16) gn_bwd_reduce_kernel<__nv_bfloat16><<<grid, threads, smem, st>>>(a);
  else gn_bwd_reduce_kernel<float><<<grid, threads, smem, st>>>(a);
  WSR_LAUNCH_OK();
  return WSR_OK;
}

extern "C" int wsr_gn_bwd_apply(const void* x, int x_dtype, int N, int HW, int C, int x_ld, const double* stats, int stats_ld,
                                const float* gamma, const float* beta, int groups, float eps, int act, const void* da,
                                int da_dtype, int da_ld, float drop_p, uint64_t drop_seed, uint32_t drop_tag, const double* red,
                                int red_ld, void* dx, int dx_dtype, int dx_ld, int accumulate, float* dgamma, float* dbeta,
                                float* colsum, int colsum_ld, void* stream) {
  GnBwdArgs a;
  int rc = gn_bwd_common(a, x, x_dtype, N, HW, C, x_ld, stats, stats_ld, gamma, beta, groups, eps, act, da, da_dtype, da_ld, drop_p,
                         drop_seed, drop_tag, const_cast<double*>(red), red_ld);
  if (rc) return rc;
  WSR_REQUIRE(dx && dx_dtype == x_dtype && dx_ld >= C, WSR_E_INVALID, "gn_bwd_apply: bad dx");
  WSR_REQUIRE((dgamma == nullptr) == (dbeta == nullptr), WSR_E_INVALID, "gn_bwd_apply: dgamma / dbeta must come together");
  WSR_REQUIRE(colsum == nullptr || colsum_ld >= C, WSR_E_INVALID, "gn_bwd_apply: colsum pitch");
  a.dx = dx; a.dx_ld = dx_ld; a.dgamma = dgamma; a.dbeta = dbeta; a.colsum = colsum; a.colsum_ld = colsum_ld;
  const int vec = gn_bwd_vec(x_dtype, C, x_ld, da_ld, dx_ld, x, da, dx);
  if (vec > 1 && (size_t)4 * C * sizeof(float) <= 48 * 1024) {
    const int CV = C / vec, PL = CV >= 256 ? 1 : 256 / CV;
    if (a.chunk < 4 * PL) a.chunk = 4 * PL < HW ? 4 * PL : HW;
    dim3 grid((HW + a.chunk - 1) / a.chunk, N);
    size_t smem = (size_t)4 * C * sizeof(float);
    cudaStream_t st = (cudaStream_t)stream;
    if (x_dtype == WSR_BF16) gn_bwd_apply_vec_kernel<__nv_bfloat16, 8><<<grid, CV * PL, smem, st>>>(a, accumulate, CV, PL);
    else gn_bwd_apply_vec_kernel<float, 4><<<grid, CV * PL, smem, st>>>(a, accumulate, CV, PL);
    WSR_LAUNCH_OK();
    return WSR_OK;
  }
  dim3 grid((HW + a.chunk - 1) / a.chunk, N);
  const int threads = C >= 256 ? 256 : ((C + 31) / 32) * 32;
  size_t smem = (size_t)4 * C * sizeof(float);
  if (smem > 48 * 1024) {
    WSR_CUDA_OK(cudaFuncSetAttribute(gn_bwd_apply_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    WSR_CUDA_OK(cudaFuncSetAttribute(gn_bwd_apply_kernel<__nv_bfloat16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  }
  cudaStream_t st = (cudaStream_t)stream;
  if (x_dtype == WSR_BF16) gn_bwd_apply_kernel<__nv_bfloat16><<<grid, threads, smem, st>>>(a, accumulate);
  else gn_bwd_apply_kernel<float><<<grid, threads, smem, st>>>(a, accumulate);
  WSR_LAUNCH_OK();
  return WSR_OK;
}

extern "C" int wsr_softmax_bwd_rows(const void* p, int p_dtype, const void* dp, int dp_dtype, int64_t rows, int cols, int64_t ld,
                                    float scale, void* ds, int ds_dtype, void* stream) {
  WSR_REQUIRE(p && dp && ds && valid_dtype(p_dtype) && valid_dtype(dp_dtype) && valid_dtype(ds_dtype) && rows > 0 && cols > 0 && ld >= cols,
              WSR_E_INVALID, "softmax_bwd_rows: bad argument");
  WSR_REQUIRE(rows <= 2147483647LL, WSR_E_UNSUPPORTED, "softmax_bwd_rows: too many rows");
  softmax_bwd_rows_kernel<<<(unsigned)rows, 128, 0, (cudaStream_t)stream>>>(p, p_dtype, dp, dp_dtype, cols, ld, scale, ds, ds_dtype);
  WSR_LAUNCH_OK();
  return WSR_OK;
}

extern "C" int wsr_noise_embed_bwd(const float* level, int R, int inner, const float* w1, const float* b1, const float* w2,
                                   int act, const float* dtemb, float* dw1, float* db1, float* dw2, float* db2, void* stream) {
  WSR_REQUIRE(level && w1 && b1 && w2 && dtemb && dw1 && db1 && dw2 && db2 && R > 0 && inner > 0 && inner % 2 == 0, WSR_E_INVALID,
              "noise_embed_bwd: bad argument");
  WSR_REQUIRE(inner <= 512, WSR_E_UNSUPPORTED, "noise_embed_bwd: inner=%d too large", inner);
  noise_embed_bwd_kernel<<<R, 256, (size_t)14 * inner * sizeof(float), (cudaStream_t)stream>>>(level, inner, w1, b1, w2, act, dtemb, dw1, db1, dw2, db2);
  WSR_LAUNCH_OK();
  return WSR_OK;
}

extern "C" int wsr_linear_rows_bwd(const float* x, int R, int K, const float* w, const float* dy, int P, float* dx, float* dw,
                                   float* db, void* stream) {
  WSR_REQUIRE(x && w && dy && R > 0 && K > 0 && P > 0, WSR_E_INVALID, "linear_rows_bwd: bad argument");
  WSR_REQUIRE(R <= 65535 && K <= 65535, WSR_E_UNSUPPORTED, "linear_rows_bwd: R=%d K=%d out of range", R, K);
  cudaStream_t st = (cudaStream_t)stream;
  if (dw) {
    const int64_t total = (int64_t)P * K;
    linear_rows_bwd_w_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(x, R, K, dy, P, dw, db);
    WSR_LAUNCH_OK();
  }
  if (dx) {
    dim3 grid(K, R);
    linear_rows_bwd_x_kernel<<<grid, 256, 0, st>>>(w, K, dy, P, dx);
    WSR_LAUNCH_OK();
  }
  return WSR_OK;
}

extern "C" int wsr_fd_gate_bwd(const void* dxin, int d_dtype, int d_ld, int ch0, const float* x, const float* ne_rows, int ne_ld,
                               int B, int C, int H, int W, const float* fc0, const float* fc2, int hidden, float* dne, int dne_ld,
                               float* dfc0, float* dfc2, void* stream) {
  WSR_REQUIRE(dxin && x && ne_rows && fc0 && fc2 && dne && dfc0 && dfc2 && valid_dtype(d_dtype), WSR_E_INVALID, "fd_gate_bwd: null pointer");
  WSR_REQUIRE(B > 0 && C > 0 && H > 0 && W > 0 && ne_ld >= W && dne_ld >= W && d_ld >= ch0 + C, WSR_E_INVALID, "fd_gate_bwd: bad shape");
  WSR_REQUIRE(C <= 32 && hidden > 0 && hidden <= 32, WSR_E_UNSUPPORTED, "fd_gate_bwd: C or hidden > 32");
  size_t smem = ((size_t)C * W + 2 * C + 2 * hidden + 4) * sizeof(float);
  WSR_REQUIRE(smem <= 48 * 1024, WSR_E_UNSUPPORTED, "fd_gate_bwd: C*W too large");
  fd_gate_bwd_kernel<<<B, 256, smem, (cudaStream_t)stream>>>(dxin, d_dtype, d_ld, ch0, x, ne_rows, ne_ld, C, H, W, fc0, fc2, hidden, dne,
                                                            dne_ld, dfc0, dfc2);
  WSR_LAUNCH_OK();
  return WSR_OK;
}

extern "C" int wsr_adam_step(float* p, const float* g, float* m, float* v, int64_t n, double lr, double beta1, double beta2, double eps,
                             double weight_decay, int step, void* stream) {
  WSR_REQUIRE(p && g && m && v && n > 0 && step > 0, WSR_E_INVALID, "adam_step: bad argument");
  const double bc1 = 1.0 - pow(beta1, (double)step);
  const double bc2 = 1.0 - pow(beta2, (double)step);
  unsigned blocks = (unsigned)((n + 255) / 256);
  if (blocks > 2368) blocks = 2368;
  adam_step_kernel<false><<<blocks, 256, 0, (cudaStream_t)stream>>>(p, g, m, v, n, (float)lr, (float)beta1, (float)beta2,
                                                                    (float)(1.0 - beta1), (float)(1.0 - beta2), (float)eps,
                                                                    (float)weight_decay, (float)bc1, (float)sqrt(bc2), nullptr, 0.f,
                                                                    0.f);
  WSR_LAUNCH_OK();
  return WSR_OK;
}

static bool ranges_overlap(const float* a, const float* b, int64_t n) { return a < b + n && b < a + n; }

extern "C" int wsr_adam_step_ema(float* p, const float* g, float* m, float* v, float* ema, int64_t n, double lr, double beta1,
                                 double beta2, double eps, double weight_decay, int step, double ema_decay, void* stream) {
  WSR_REQUIRE(p && g && m && v && ema && n > 0 && step > 0, WSR_E_INVALID, "adam_step_ema: bad argument");
  WSR_REQUIRE(ema_decay >= 0.0 && ema_decay < 1.0, WSR_E_INVALID, "adam_step_ema: ema_decay %g outside [0, 1)", ema_decay);
  WSR_REQUIRE(!ranges_overlap(ema, p, n) && !ranges_overlap(ema, g, n) && !ranges_overlap(ema, m, n) && !ranges_overlap(ema, v, n),
              WSR_E_INVALID, "adam_step_ema: ema overlaps p, g, m or v");
  const double bc1 = 1.0 - pow(beta1, (double)step);
  const double bc2 = 1.0 - pow(beta2, (double)step);
  unsigned blocks = (unsigned)((n + 255) / 256);
  if (blocks > 2368) blocks = 2368;
  adam_step_kernel<true><<<blocks, 256, 0, (cudaStream_t)stream>>>(p, g, m, v, n, (float)lr, (float)beta1, (float)beta2,
                                                                   (float)(1.0 - beta1), (float)(1.0 - beta2), (float)eps,
                                                                   (float)weight_decay, (float)bc1, (float)sqrt(bc2), ema,
                                                                   (float)ema_decay, (float)(1.0 - ema_decay));
  WSR_LAUNCH_OK();
  return WSR_OK;
}
