// elementwise.cu -- HBM-bound kernels of the path: layout/packing, GroupNorm(+activation), row softmax, noise-level
// embedding, DDPM process updates.  All are coalesced over the NHWC channel axis and vectorised to 16 bytes where
// the pitch allows it.
#include "common.cuh"
#include "philox.cuh"

namespace wsr {

// ------------------------------------------------------------------------------------------------------------------
// layout
// ------------------------------------------------------------------------------------------------------------------
__global__ void nchw_to_nhwc_kernel(const float* __restrict__ src, int C, int64_t HW, void* dst, int dt, int ld, int64_t total) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  int c = (int)(i % C);
  int64_t np = i / C;           // n*HW + p
  int64_t n = np / HW, p = np - n * HW;
  st_dt(dst, np * ld + c, dt, src[(n * C + c) * HW + p]);
}

__global__ void nhwc_to_nchw_kernel(const void* src, int dt, int ld, int C, int64_t HW, float* __restrict__ dst, int64_t total) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  int64_t p = i % HW;
  int64_t nc = i / HW;
  int64_t n = nc / C; int c = (int)(nc - n * C);
  dst[i] = ld_dt(src, (n * HW + p) * ld + c, dt);
}

__global__ void pack_conv_weight_kernel(const float* __restrict__ w, int Cout, int Cin, int taps, void* dst, int dt,
                                        int Cout_pad, int Cin_pad, int64_t total) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  int ci = (int)(i % Cin_pad);
  int64_t r = i / Cin_pad;
  int co = (int)(r % Cout_pad);
  int t = (int)(r / Cout_pad);
  float v = (co < Cout && ci < Cin) ? w[((int64_t)co * Cin + ci) * taps + t] : 0.f;
  st_dt(dst, i, dt, v);
}

// vertical-tap-merge pack: dst[(kx*192 + b*64 + co)*Cin_pad + ci] = w[co][ci][ky = 2 - b][kx]
__global__ void pack_conv_weight_vmerge_kernel(const float* __restrict__ w, int Cout, int Cin, void* dst, int dt, int Cin_pad, int64_t total) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  int ci = (int)(i % Cin_pad);
  int64_t r = i / Cin_pad;
  int row = (int)(r % 192);
  int kx = (int)(r / 192);
  int b = row / 64, co = row % 64;
  float v = (co < Cout && ci < Cin) ? w[((int64_t)co * Cin + ci) * 9 + (2 - b) * 3 + kx] : 0.f;
  st_dt(dst, i, dt, v);
}

// merged taps of upsample+conv: row sets  py=0: a=0 -> {ky 0}, a=1 -> {ky 1,2};  py=1: a=0 -> {ky 0,1}, a=1 -> {ky 2}
__global__ void pack_upsample_weight_kernel(const float* __restrict__ w, int Cout, int Cin, void* dst, int dt, int Cout_pad,
                                            int Cin_pad, int64_t total) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  int ci = (int)(i % Cin_pad);
  int64_t r = i / Cin_pad;
  int co = (int)(r % Cout_pad);
  int t = (int)(r / Cout_pad);           // phase*4 + a*2 + b
  int ph = t >> 2, a = (t >> 1) & 1, b = t & 1;
  int py = ph >> 1, px = ph & 1;
  float v = 0.f;
  if (co < Cout && ci < Cin) {
    int ky0 = py == 0 ? (a == 0 ? 0 : 1) : (a == 0 ? 0 : 2), ky1 = py == 0 ? (a == 0 ? 0 : 2) : (a == 0 ? 1 : 2);
    int kx0 = px == 0 ? (b == 0 ? 0 : 1) : (b == 0 ? 0 : 2), kx1 = px == 0 ? (b == 0 ? 0 : 2) : (b == 0 ? 1 : 2);
    const float* wp = w + ((int64_t)co * Cin + ci) * 9;
    for (int ky = ky0; ky <= ky1; ++ky)
      for (int kx = kx0; kx <= kx1; ++kx) v += wp[ky * 3 + kx];
  }
  st_dt(dst, i, dt, v);
}

__global__ void pack_convT_weight_kernel(const float* __restrict__ w, int Cin, int Cout, int taps, void* dst, int dt, int64_t total) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;   // dst index = (t*Cout + co)*Cin + ci
  if (i >= total) return;
  int ci = (int)(i % Cin);
  int64_t r = i / Cin;
  int co = (int)(r % Cout);
  int t = (int)(r / Cout);
  st_dt(dst, i, dt, w[((int64_t)ci * Cout + co) * taps + t]);
}

// One launch re-packs EVERY weight of a plan after an optimizer step (the training loop's refresh): a device-side job
// table lists (source parameter, destination buffer, layout kind); one thread owns one (row, column) pair of one job
// and writes all of its taps, so the 36-byte tap vector of the OIHW source is read once and every destination plane is
// written coalesced along the column index.
__device__ __forceinline__ int upsample_dgrad_lo(int r) { return r == 0 ? 2 : (r == 1 ? 1 : 0); }          // r = row offset + 1
__device__ __forceinline__ int upsample_dgrad_hi(int r) { return r == 0 ? 2 : (r == 1 ? 2 : (r == 2 ? 1 : 0)); }

__global__ void repack_batch_kernel(const WsrPackJob* __restrict__ jobs, int njobs, int64_t total) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    int lo = 0, hi = njobs - 1;
    while (lo < hi) {
      int mid = (lo + hi + 1) >> 1;
      if (jobs[mid].first_unit <= i) lo = mid; else hi = mid - 1;
    }
    const WsrPackJob j = jobs[lo];
    int64_t u = i - j.first_unit;
    if (j.kind == WSR_PACK_COPY) {
      float v = j.src[u];
      if (j.src2) v += j.src2[u];
      st_dt(j.dst, u, j.dst_dtype, v);
      continue;
    }
    const int ci = (int)(u % j.Cin_pad), co = (int)(u / j.Cin_pad);
    const bool valid = co < j.Cout && ci < j.Cin;
    const int T = j.taps;
    const float* wp = j.src + (j.transposed ? ((int64_t)ci * j.Cout + co) : ((int64_t)co * j.Cin + ci)) * T;
    const int64_t plane = (int64_t)j.Cout_pad * j.Cin_pad;
    const int64_t o = (int64_t)co * j.Cin_pad + ci;
    if (j.kind == WSR_PACK_CONV) {
      for (int t = 0; t < T; ++t) st_dt(j.dst, t * plane + o, j.dst_dtype, valid ? wp[j.transposed ? T - 1 - t : t] : 0.f);
    } else {
      float w9[9];
#pragma unroll
      for (int t = 0; t < 9; ++t) w9[t] = valid ? wp[t] : 0.f;
      if (j.kind == WSR_PACK_VMERGE) {            // dst[(kx*192 + b*64 + co)*Cin_pad + ci] = w'[co][ci][ky = 2-b][kx]
#pragma unroll
        for (int kx = 0; kx < 3; ++kx)
#pragma unroll
          for (int b = 0; b < 3; ++b) {
            int t = (2 - b) * 3 + kx;
            st_dt(j.dst, ((int64_t)(kx * 192 + b * 64 + co)) * j.Cin_pad + ci, j.dst_dtype, w9[j.transposed ? 8 - t : t]);
          }
      } else if (j.kind == WSR_PACK_UPSAMPLE) {   // see pack_upsample_weight_kernel
#pragma unroll
        for (int t = 0; t < 16; ++t) {
          int ph = t >> 2, a = (t >> 1) & 1, b = t & 1, py = ph >> 1, px = ph & 1;
          int ky0 = py == 0 ? (a == 0 ? 0 : 1) : (a == 0 ? 0 : 2), ky1 = py == 0 ? (a == 0 ? 0 : 2) : (a == 0 ? 1 : 2);
          int kx0 = px == 0 ? (b == 0 ? 0 : 1) : (b == 0 ? 0 : 2), kx1 = px == 0 ? (b == 0 ? 0 : 2) : (b == 0 ? 1 : 2);
          float v = 0.f;
          for (int ky = ky0; ky <= ky1; ++ky)
            for (int kx = kx0; kx <= kx1; ++kx) v += w9[ky * 3 + kx];
          st_dt(j.dst, t * plane + o, j.dst_dtype, v);
        }
      } else {                                    // WSR_PACK_UPSAMPLE_DGRAD: 4x4 taps, tap (r, s) = sum of the 3x3 taps reaching it
#pragma unroll
        for (int t = 0; t < 16; ++t) {
          int r = t >> 2, s = t & 3;
          float v = 0.f;
          for (int ky = upsample_dgrad_lo(r); ky <= upsample_dgrad_hi(r); ++ky)
            for (int kx = upsample_dgrad_lo(s); kx <= upsample_dgrad_hi(s); ++kx) v += w9[ky * 3 + kx];
          st_dt(j.dst, t * plane + o, j.dst_dtype, v);
        }
      }
    }
  }
}

__global__ void cast_kernel(const void* src, int sdt, void* dst, int ddt, int64_t n) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) st_dt(dst, i, ddt, ld_dt(src, i, sdt));
}

template <typename T>
__global__ void upsample2x_kernel(const T* __restrict__ x, int H, int W, int C, int x_ld, T* __restrict__ y, int y_ld, int64_t total) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;   // over N*2H*2W*C
  if (i >= total) return;
  int c = (int)(i % C);
  int64_t r = i / C;
  int ox = (int)(r % (2 * W)); r /= (2 * W);
  int oy = (int)(r % (2 * H));
  int64_t n = r / (2 * H);
  y[((n * 2 * H + oy) * 2 * W + ox) * y_ld + c] = x[((n * H + (oy >> 1)) * W + (ox >> 1)) * x_ld + c];
}

__global__ void axpby_kernel(const void* x, int xdt, int x_ld, float a, const void* z, int zdt, int z_ld, float b,
                             void* y, int ydt, int y_ld, int C, int64_t total) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  int c = (int)(i % C);
  int64_t p = i / C;
  st_dt(y, p * y_ld + c, ydt, a * ld_dt(x, p * x_ld + c, xdt) + b * ld_dt(z, p * z_ld + c, zdt));
}

// ------------------------------------------------------------------------------------------------------------------
// GroupNorm: per-(image, channel) sums, then normalise (+ activation)
// thread layout: blockDim = CV * PL; thread t owns channel vector t % CV and pixel lane t / CV.
// ------------------------------------------------------------------------------------------------------------------
template <typename T, int VEC>
__global__ void gn_stats_kernel(const T* __restrict__ x, int HW, int C, int ld, int CV, int PL, int chunk, double* __restrict__ stats, int stats_ld) {
  extern __shared__ float sm[];   // [PL][C][2]
  const int n = blockIdx.y;
  const int cv = threadIdx.x % CV, pl = threadIdx.x / CV;
  const int p0 = blockIdx.x * chunk;
  const int p1 = min(HW, p0 + chunk);
  float s[VEC], q[VEC];
#pragma unroll
  for (int i = 0; i < VEC; ++i) { s[i] = 0.f; q[i] = 0.f; }
  const T* base = x + (int64_t)n * HW * ld + cv * VEC;
  int p = p0 + pl;
  for (; p + 3 * PL < p1; p += 4 * PL) {          // four independent 16-byte loads in flight per thread
    float v[4][VEC];
#pragma unroll
    for (int u = 0; u < 4; ++u) VecLoad<T, VEC>::ld(base + (int64_t)(p + u * PL) * ld, v[u]);
#pragma unroll
    for (int u = 0; u < 4; ++u)
#pragma unroll
      for (int i = 0; i < VEC; ++i) { s[i] += v[u][i]; q[i] = fmaf(v[u][i], v[u][i], q[i]); }
  }
  for (; p < p1; p += PL) {
    float v[VEC];
    VecLoad<T, VEC>::ld(base + (int64_t)p * ld, v);
#pragma unroll
    for (int i = 0; i < VEC; ++i) { s[i] += v[i]; q[i] = fmaf(v[i], v[i], q[i]); }
  }
#pragma unroll
  for (int i = 0; i < VEC; ++i) {
    sm[(pl * C + cv * VEC + i) * 2 + 0] = s[i];
    sm[(pl * C + cv * VEC + i) * 2 + 1] = q[i];
  }
  __syncthreads();
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    double a = 0.0, b = 0.0;
    for (int l = 0; l < PL; ++l) { a += (double)sm[(l * C + c) * 2]; b += (double)sm[(l * C + c) * 2 + 1]; }
    atomicAdd(&stats[(int64_t)n * stats_ld + c * 2 + 0], a);
    atomicAdd(&stats[(int64_t)n * stats_ld + c * 2 + 1], b);
  }
}

// DROP: training-mode dropout after the activation (nn_modules/resnet.py:23): y *= mask / (1 - p), mask from Philox
// (seed, tag, logical element index (n*HW + p)*C + c) so that the backward pass can regenerate it.
template <typename TI, typename TO, int VEC, bool DROP>
__global__ void gn_apply_kernel(const TI* __restrict__ x, int HW, int C, int ld, int CV, int PL, int chunk,
                                const double* __restrict__ stats, int stats_ld, const float* __restrict__ gamma,
                                const float* __restrict__ beta, int groups, float eps, int act, TO* __restrict__ y, int y_ld,
                                float drop_p, uint64_t drop_seed, uint32_t drop_tag) {
  extern __shared__ float sm[];   // scale[C], shift[C], then (mean, rstd) per group
  // Block -> (image, pixel chunk) in natural order.  Walking the ranges the producing convolution's CTAs wrote back to front, to
  // read their L2-resident tails first, MEASURED no faster on B200 (profiles/r02_gn_order_ab.txt): the 65 gn_apply launches of a B = 64
  // step take 3.09 ms that way vs 3.03 ms in natural order, the whole step 16.64 vs 16.56 ms (3.53 vs 3.51 ms at B = 8) -- the
  // write-back L2 does not keep the producer's tail lines resident the way an LRU read cache would.
  const int n = blockIdx.y;
  const int chunk_idx = blockIdx.x;
  const int cpg = C / groups;
  float* gm = sm + 2 * C;
  pdl_launch_dependents();        // programmatic dependent launch (common.cuh): the statistics come from the preceding convolution
  pdl_wait();
  // group moments first (one thread per group sums its cpg channel statistics), then per-channel scale / shift: the
  // per-channel version re-summed the whole group for every channel (2 * cpg double loads each; cpg = 32 at C = 1024)
  for (int g = threadIdx.x; g < groups; g += blockDim.x) {
    double a = 0.0, b = 0.0;
    for (int j = 0; j < cpg; ++j) { a += stats[(int64_t)n * stats_ld + (g * cpg + j) * 2]; b += stats[(int64_t)n * stats_ld + (g * cpg + j) * 2 + 1]; }
    // sums and the E[x^2] - mean^2 cancellation stay in double; the reciprocal square root is taken in fp32 in bf16 mode
    const double inv_cnt = 1.0 / ((double)cpg * HW);
    const double mean = a * inv_cnt;
    double var = b * inv_cnt - mean * mean;
    if (var < 0.0) var = 0.0;
    gm[2 * g] = (float)mean;
    gm[2 * g + 1] = sizeof(TI) == 4 ? (float)(1.0 / sqrt(var + (double)eps)) : rsqrtf((float)var + eps);
  }
  __syncthreads();
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    const int g = c / cpg;
    const float sc = gamma[c] * gm[2 * g + 1];
    sm[c] = sc;
    sm[C + c] = beta[c] - gm[2 * g] * sc;
  }
  __syncthreads();
  const int cv = threadIdx.x % CV, pl = threadIdx.x / CV;
  const int p0 = chunk_idx * chunk;
  const int p1 = min(HW, p0 + chunk);
  float sc[VEC], sh[VEC];
#pragma unroll
  for (int i = 0; i < VEC; ++i) { sc[i] = sm[cv * VEC + i]; sh[i] = sm[C + cv * VEC + i]; }
  const TI* xb = x + (int64_t)n * HW * ld + cv * VEC;
  TO* yb = y + (int64_t)n * HW * y_ld + cv * VEC;
  int p = p0 + pl;
  for (; p + 3 * PL < p1; p += 4 * PL) {          // four independent 16-byte loads in flight per thread
    // the loaded vectors stay RAW (4 registers each for bf16) until their turn: widening all four up front cost 32 live fp32
    // registers, 72 per thread and 3 resident blocks per SM (ncu: 33 % achieved occupancy, 61 % of the DRAM peak)
    typename VecLoad<TI, VEC>::Raw raw[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) raw[u] = VecLoad<TI, VEC>::ldraw(xb + (int64_t)(p + u * PL) * ld);
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      float v[VEC];
      VecLoad<TI, VEC>::widen(raw[u], v);
#pragma unroll
      for (int i = 0; i < VEC; ++i) {
        const float t = fmaf(v[i], sc[i], sh[i]);
        v[i] = (sizeof(TO) == 2 && act == WSR_ACT_SWISH) ? swish_fast(t) : apply_act(t, act);
      }
      if constexpr (DROP) {
        float m[VEC];
        dropout_scale<VEC>(drop_seed, drop_tag, ((uint64_t)n * HW + (uint64_t)(p + u * PL)) * C + (uint64_t)cv * VEC, drop_p, m);
#pragma unroll
        for (int i = 0; i < VEC; ++i) v[i] *= m[i];
      }
      VecLoad<TO, VEC>::st(yb + (int64_t)(p + u * PL) * y_ld, v);
    }
  }
  for (; p < p1; p += PL) {
    float v[VEC];
    VecLoad<TI, VEC>::ld(xb + (int64_t)p * ld, v);
#pragma unroll
    for (int i = 0; i < VEC; ++i) {
      const float t = fmaf(v[i], sc[i], sh[i]);
      v[i] = (sizeof(TO) == 2 && act == WSR_ACT_SWISH) ? swish_fast(t) : apply_act(t, act);
    }
    if constexpr (DROP) {
      float m[VEC];
      dropout_scale<VEC>(drop_seed, drop_tag, ((uint64_t)n * HW + (uint64_t)p) * C + (uint64_t)cv * VEC, drop_p, m);
#pragma unroll
      for (int i = 0; i < VEC; ++i) v[i] *= m[i];
    }
    VecLoad<TO, VEC>::st(yb + (int64_t)p * y_ld, v);
  }
}

// (scale, shift) per (image, channel): a = x * scale + shift  ==  GroupNorm(x) * gamma + beta
__global__ void gn_finalize_kernel(const double* __restrict__ stats, int stats_ld, int HW, int C, int groups, float eps,
                                   const float* __restrict__ gamma, const float* __restrict__ beta, float2* __restrict__ tab, int tab_ld) {
  const int n = blockIdx.x;
  const int cpg = C / groups;
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    const int g0 = (c / cpg) * cpg;
    double a = 0.0, b = 0.0;
    for (int j = 0; j < cpg; ++j) { a += stats[(int64_t)n * stats_ld + (g0 + j) * 2]; b += stats[(int64_t)n * stats_ld + (g0 + j) * 2 + 1]; }
    const double cnt = (double)cpg * HW;
    const double mean = a / cnt;
    double var = b / cnt - mean * mean;
    if (var < 0.0) var = 0.0;
    const float rstd = (float)(1.0 / sqrt(var + (double)eps));
    const float sc = gamma[c] * rstd;
    tab[(int64_t)n * tab_ld + c] = make_float2(sc, beta[c] - (float)mean * sc);
  }
}

struct GnGeom { int vec, CV, PL, chunk, threads; };
static GnGeom gn_geom(int dt, int C, int ld, int ld2, const void* p, const void* p2) {
  GnGeom g;
  int want = dt == WSR_BF16 ? 8 : 4;
  bool ok = (C % want == 0) && (ld % want == 0) && (ld2 % want == 0) && (((uintptr_t)p & 15) == 0) && (((uintptr_t)p2 & 15) == 0);
  g.vec = ok ? want : 1;
  g.CV = C / g.vec;
  while (g.CV > 1024) { g.vec = 0; break; }
  g.PL = g.CV >= 256 ? 1 : 256 / g.CV;
  g.threads = g.CV * g.PL;
  g.chunk = g.PL * 64;
  return g;
}

// ------------------------------------------------------------------------------------------------------------------
// row softmax
// ------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
template <int NT> __device__ __forceinline__ float block_max(float v, float* red) {
  v = warp_max(v);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  float r = red[0];
#pragma unroll
  for (int i = 1; i < NT / 32; ++i) r = fmaxf(r, red[i]);
  __syncthreads();
  return r;
}
template <int NT> __device__ __forceinline__ float block_sum(float v, float* red) {
  v = warp_sum(v);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  float r = 0.f;
#pragma unroll
  for (int i = 0; i < NT / 32; ++i) r += red[i];
  __syncthreads();
  return r;
}

__global__ void __launch_bounds__(128) softmax_rows_kernel(const void* s, int sdt, int cols, int64_t s_ld, float scale,
                                                          void* p, int pdt, int64_t p_ld) {
  __shared__ float red[4];
  const int64_t r = blockIdx.x;
  float mx = -INFINITY;
  for (int c = threadIdx.x; c < cols; c += 128) mx = fmaxf(mx, ld_dt(s, r * s_ld + c, sdt) * scale);
  mx = block_max<128>(mx, red);
  float sum = 0.f;
  for (int c = threadIdx.x; c < cols; c += 128) sum += __expf(ld_dt(s, r * s_ld + c, sdt) * scale - mx);
  sum = block_sum<128>(sum, red);
  float inv = 1.f / sum;
  for (int c = threadIdx.x; c < cols; c += 128)
    st_dt(p, r * p_ld + c, pdt, __expf(ld_dt(s, r * s_ld + c, sdt) * scale - mx) * inv);
}

// One WARP per row for the attention shapes of the sampler (fp32 scores, cols = NV * 128 <= 1024): the row is read ONCE into registers
// with 16-byte loads (the block-per-row kernel above reads it three times with 4-byte loads and pays two block reductions per row:
// 2.4 TB/s of algorithmic traffic), maxima and sums by warp shuffles, probabilities stored as packed bf16 (8 bytes per lane) or fp32.
template <int NV>
__global__ void __launch_bounds__(256) softmax_rows_warp_kernel(const float* __restrict__ s, int64_t s_ld, float scale, void* __restrict__ p,
                                                               int pdt, int64_t p_ld, int64_t rows) {
  const int64_t r = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (r >= rows) return;
  const int lane = threadIdx.x & 31;
  const float4* sp = (const float4*)(s + r * s_ld) + lane;
  float4 v[NV];
#pragma unroll
  for (int i = 0; i < NV; ++i) v[i] = __ldcs(sp + i * 32);
  float mx = -INFINITY;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    v[i].x *= scale; v[i].y *= scale; v[i].z *= scale; v[i].w *= scale;
    mx = fmaxf(mx, fmaxf(fmaxf(v[i].x, v[i].y), fmaxf(v[i].z, v[i].w)));
  }
  mx = warp_max(mx);
  float sum = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    v[i].x = __expf(v[i].x - mx); v[i].y = __expf(v[i].y - mx); v[i].z = __expf(v[i].z - mx); v[i].w = __expf(v[i].w - mx);
    sum += (v[i].x + v[i].y) + (v[i].z + v[i].w);
  }
  sum = warp_sum(sum);
  const float inv = 1.f / sum;
  if (pdt == WSR_BF16) {
    uint2* pp = (uint2*)((__nv_bfloat16*)p + r * p_ld) + lane;
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      uint2 u;
      *(__nv_bfloat162*)&u.x = __floats2bfloat162_rn(v[i].x * inv, v[i].y * inv);
      *(__nv_bfloat162*)&u.y = __floats2bfloat162_rn(v[i].z * inv, v[i].w * inv);
      pp[i * 32] = u;
    }
  } else {
    float4* pp = (float4*)((float*)p + r * p_ld) + lane;
#pragma unroll
    for (int i = 0; i < NV; ++i) pp[i * 32] = make_float4(v[i].x * inv, v[i].y * inv, v[i].z * inv, v[i].w * inv);
  }
}

// ------------------------------------------------------------------------------------------------------------------
// noise-level embedding
// ------------------------------------------------------------------------------------------------------------------
__global__ void noise_embed_kernel(const float* __restrict__ level, int inner, const float* __restrict__ w1,
                                   const float* __restrict__ b1, const float* __restrict__ w2,
                                   const float* __restrict__ b2, int act, float* __restrict__ temb) {
  extern __shared__ float sm[];   // enc[inner], hid[4*inner]
  float* enc = sm;
  float* hid = sm + inner;
  const int r = blockIdx.x;
  const float lv = level[r];
  const int half = inner / 2;
  for (int k = threadIdx.x; k < half; k += blockDim.x) {
    float step = (float)k / (float)half;
    float arg = lv * expf(-logf(1e4f) * step);
    enc[k] = sinf(arg);
    enc[half + k] = cosf(arg);
  }
  __syncthreads();
  for (int o = threadIdx.x; o < 4 * inner; o += blockDim.x) {
    float a = b1[o];
    for (int k = 0; k < inner; ++k) a = fmaf(w1[(int64_t)o * inner + k], enc[k], a);
    hid[o] = apply_act(a, act);
  }
  __syncthreads();
  for (int o = threadIdx.x; o < inner; o += blockDim.x) {
    float a = b2[o];
    for (int k = 0; k < 4 * inner; ++k) a = fmaf(w2[(int64_t)o * 4 * inner + k], hid[k], a);
    temb[(int64_t)r * inner + o] = a;
  }
}

__global__ void linear_rows_kernel(const float* __restrict__ x, int K, const float* __restrict__ w,
                                   const float* __restrict__ bias, int P, float* __restrict__ y) {
  extern __shared__ float xs[];   // x row
  const int r = blockIdx.y;
  for (int k = threadIdx.x; k < K; k += blockDim.x) xs[k] = x[(int64_t)r * K + k];
  __syncthreads();
  int o = blockIdx.x * blockDim.x + threadIdx.x;
  if (o >= P) return;
  float a = bias ? bias[o] : 0.f;
  for (int k = 0; k < K; ++k) a = fmaf(w[(int64_t)o * K + k], xs[k], a);
  y[(int64_t)r * P + o] = a;
}

// ------------------------------------------------------------------------------------------------------------------
// DDPM process
// ------------------------------------------------------------------------------------------------------------------
// four standard normals for element group `grp` of stream (seed, tag)
__device__ __forceinline__ void randn4(uint64_t seed, uint32_t tag, uint64_t grp, float (&z)[4]) {
  uint32_t c[4] = {(uint32_t)grp, (uint32_t)(grp >> 32), tag, 0x5752u};
  philox4x32_10(c, (uint32_t)seed, (uint32_t)(seed >> 32));
  const float s = 2.3283064365386963e-10f;   // 2^-32
  float u0 = ((float)c[0] + 0.5f) * s, u1 = ((float)c[1] + 0.5f) * s;
  float u2 = ((float)c[2] + 0.5f) * s, u3 = ((float)c[3] + 0.5f) * s;
  float r0 = sqrtf(-2.f * __logf(u0)), r1 = sqrtf(-2.f * __logf(u2));
  float s0, c0, s1, c1;
  __sincosf(6.283185307179586f * u1, &s0, &c0);
  __sincosf(6.283185307179586f * u3, &s1, &c1);
  z[0] = r0 * c0; z[1] = r0 * s0; z[2] = r1 * c1; z[3] = r1 * s1;
}

// Philox key and member-local group of the 4-element group g: the plain stream (key = seed, group g), or the member-keyed stream of
// an ensemble batch (member m = g / member_groups draws from key member_keys[m] at group g - m * member_groups), so that member m's
// slice is exactly the plain stream of key member_keys[m] over that slice alone.
template <bool MK>
__device__ __forceinline__ uint64_t noise_key(uint64_t seed, const uint64_t* __restrict__ member_keys, int64_t member_groups, int64_t& g) {
  if constexpr (MK) {
    const int64_t m = g / member_groups;
    g -= m * member_groups;
    return __ldg((const unsigned long long*)member_keys + m);
  } else {
    (void)member_keys; (void)member_groups;
    return seed;
  }
}

// MS = false: the DDPM / DDIM step, tables (c_recip, c_recipm1, coef1, coef2, logvar), noise from the chain z or Philox.
// MS = true: the multistep (DPM-Solver++(2M)) step, tables (c_recip, c_recipm1, c_x0, c_x, c_prev): x_out = c_x0 x0 + c_x x + c_prev hist,
// then hist <- x0 (clamped); no noise.  hist is not read when c_prev == 0 (first and final steps), so its initial contents never matter.
template <bool MK, bool MS>
__global__ void sampler_step_kernel(const float* x, const void* eps, int edt, const float* __restrict__ z, int64_t z_stride,
                                    uint64_t seed, const uint64_t* __restrict__ member_keys, int64_t member_groups, float* __restrict__ hist,
                                    const float* __restrict__ tab, int T, const int* __restrict__ t_dev, int clip, float* xo, int64_t n) {
  const int t = *t_dev;
  if (!MS && z) z += (int64_t)(T - t) * z_stride;
  const float c_recip = tab[t], c_recipm1 = tab[T + t], coef1 = tab[2 * T + t], coef2 = tab[3 * T + t];
  const float sigma = !MS && t > 0 ? __expf(0.5f * tab[4 * T + t]) : 0.f;
  const float c_prev = MS ? tab[4 * T + t] : 0.f;
  int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;   // group of 4 elements
  int64_t i0 = g * 4;
  if (i0 >= n) return;
  float zz[4] = {0.f, 0.f, 0.f, 0.f};
  if (!MS && t > 0) {
    if (z) {
#pragma unroll
      for (int j = 0; j < 4; ++j) if (i0 + j < n) zz[j] = z[i0 + j];
    } else {
      int64_t lg = g;
      const uint64_t key = noise_key<MK>(seed, member_keys, member_groups, lg);
      randn4(key, (uint32_t)t, (uint64_t)lg, zz);
    }
  }
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    int64_t i = i0 + j;
    if (i >= n) break;
    float xv = x[i];
    float x0 = c_recip * xv - c_recipm1 * ld_dt(eps, i, edt);
    if (clip) x0 = fminf(1.f, fmaxf(-1.f, x0));
    if constexpr (MS) {
      float o = coef1 * x0 + coef2 * xv;
      if (c_prev != 0.f) o += c_prev * hist[i];
      hist[i] = x0;
      xo[i] = o;
    } else {
      xo[i] = coef1 * x0 + coef2 * xv + sigma * zz[j];
    }
  }
}

__global__ void step_counter_add_kernel(int* t, int delta) { *t += delta; }

__global__ void broadcast_row_kernel(const float* __restrict__ table, int P, const int* __restrict__ row_index, float* __restrict__ out) {
  const float* src = table + (int64_t)(*row_index) * P;
  float* dst = out + (int64_t)blockIdx.y * P;
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < P) dst[i] = src[i];
}

template <bool MK>
__global__ void randn_kernel(float* out, int64_t n, uint64_t seed, const uint64_t* __restrict__ member_keys, int64_t member_groups,
                             uint32_t tag) {
  int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g * 4 >= n) return;
  float z[4];
  int64_t lg = g;
  const uint64_t key = noise_key<MK>(seed, member_keys, member_groups, lg);
  randn4(key, tag, (uint64_t)lg, z);
#pragma unroll
  for (int j = 0; j < 4; ++j) if (g * 4 + j < n) out[g * 4 + j] = z[j];
}

__global__ void q_sample_kernel(const float* __restrict__ hr, const float* __restrict__ sr, const float* __restrict__ noise,
                                const float* __restrict__ a, int64_t per, float* __restrict__ xn, int64_t n) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float av = a[i / per];
  xn[i] = av * (hr[i] - sr[i]) + sqrtf(1.f - av * av) * noise[i];
}

__global__ void __launch_bounds__(256) noise_loss_kernel(const float* __restrict__ noise, const float* __restrict__ eps,
                                                         int64_t n, int l2, double* loss, float* grad, float scale) {
  __shared__ float red[8];
  float acc = 0.f;
  for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (int64_t)gridDim.x * 256) {
    float d = noise[i] - eps[i];
    acc += l2 ? d * d : fabsf(d);
    if (grad) grad[i] = l2 ? -2.f * d * scale : (d > 0.f ? -scale : (d < 0.f ? scale : 0.f));
  }
  float tot = block_sum<256>(acc, red);
  if (threadIdx.x == 0) atomicAdd(loss, (double)tot);
}

}  // namespace wsr

using namespace wsr;
static inline unsigned blocks_for(int64_t n, int t) { return (unsigned)((n + t - 1) / t); }

extern "C" int wsr_nchw_to_nhwc(const float* src, int N, int C, int H, int W, void* dst, int dst_dtype, int dst_ld, void* stream) {
  WSR_REQUIRE(src && dst && valid_dtype(dst_dtype) && N > 0 && C > 0 && H > 0 && W > 0 && dst_ld >= C, WSR_E_INVALID, "nchw_to_nhwc: bad argument");
  int64_t total = (int64_t)N * C * H * W;
  nchw_to_nhwc_kernel<<<blocks_for(total, 256), 256, 0, (cudaStream_t)stream>>>(src, C, (int64_t)H * W, dst, dst_dtype, dst_ld, total);
  WSR_LAUNCH_OK();
  return WSR_OK;
}

extern "C" int wsr_nhwc_to_nchw(const void* src, int src_dtype, int src_ld, int N, int C, int H, int W, float* dst, void* stream) {
  WSR_REQUIRE(src && dst && valid_dtype(src_dtype) && N > 0 && C > 0 && H > 0 && W > 0 && src_ld >= C, WSR_E_INVALID, "nhwc_to_nchw: bad argument");
  int64_t total = (int64_t)N * C * H * W;
  nhwc_to_nchw_kernel<<<blocks_for(total, 256), 256, 0, (cudaStream_t)stream>>>(src, src_dtype, src_ld, C, (int64_t)H * W, dst, total);
  WSR_LAUNCH_OK();
  return WSR_OK;
}

extern "C" int wsr_pack_conv_weight(const float* w, int Cout, int Cin, int KH, int KW, void* dst, int dst_dtype,
                                    int Cout_pad, int Cin_pad, void* stream) {
  WSR_REQUIRE(w && dst && valid_dtype(dst_dtype) && Cout > 0 && Cin > 0 && KH > 0 && KW > 0 && Cout_pad >= Cout && Cin_pad >= Cin,
              WSR_E_INVALID, "pack_conv_weight: bad argument");
  int64_t total = (int64_t)KH * KW * Cout_pad * Cin_pad;
  pack_conv_weight_kernel<<<blocks_for(total, 256), 256, 0, (cudaStream_t)stream>>>(w, Cout, Cin, KH * KW, dst, dst_dtype, Cout_pad, Cin_pad, total);
  WSR_LAUNCH_OK();
  return WSR_OK;
}

extern "C" int wsr_pack_conv_weight_vmerge(const float* w, int Cout, int Cin, void* dst, int dst_dtype, int Cin_pad, void* stream) {
  WSR_REQUIRE(w && dst && valid_dtype(dst_dtype) && Cout > 0 && Cout <= 64 && Cin > 0 && Cin_pad >= Cin, WSR_E_INVALID, "pack_conv_weight_vmerge: bad argument");
  int64_t total = (int64_t)3 * 192 * Cin_pad;
  pack_conv_weight_vmerge_kernel<<<blocks_for(total, 256), 256, 0, (cudaStream_t)stream>>>(w, Cout, Cin, dst, dst_dtype, Cin_pad, total);
  WSR_LAUNCH_OK();
  return WSR_OK;
}

extern "C" int wsr_pack_upsample_weight(const float* w, int Cout, int Cin, void* dst, int dst_dtype, int Cout_pad, int Cin_pad,
                                        void* stream) {
  WSR_REQUIRE(w && dst && valid_dtype(dst_dtype) && Cout > 0 && Cin > 0 && Cout_pad >= Cout && Cin_pad >= Cin, WSR_E_INVALID,
              "pack_upsample_weight: bad argument");
  int64_t total = (int64_t)16 * Cout_pad * Cin_pad;
  pack_upsample_weight_kernel<<<blocks_for(total, 256), 256, 0, (cudaStream_t)stream>>>(w, Cout, Cin, dst, dst_dtype, Cout_pad, Cin_pad, total);
  WSR_LAUNCH_OK();
  return WSR_OK;
}

extern "C" int wsr_pack_convT_weight(const float* w, int Cin, int Cout, int KH, int KW, void* dst, int dst_dtype, void* stream) {
  WSR_REQUIRE(w && dst && valid_dtype(dst_dtype) && Cout > 0 && Cin > 0 && KH > 0 && KW > 0, WSR_E_INVALID, "pack_convT_weight: bad argument");
  int64_t total = (int64_t)KH * KW * Cout * Cin;
  pack_convT_weight_kernel<<<blocks_for(total, 256), 256, 0, (cudaStream_t)stream>>>(w, Cin, Cout, KH * KW, dst, dst_dtype, total);
  WSR_LAUNCH_OK();
  return WSR_OK;
}

extern "C" int wsr_repack_batch(const WsrPackJob* jobs_device, int njobs, int64_t total_units, void* stream) {
  WSR_REQUIRE(jobs_device && njobs > 0 && total_units > 0, WSR_E_INVALID, "repack_batch: bad argument");
  int64_t blocks = (total_units + 255) / 256;
  if (blocks > 148 * 64) blocks = 148 * 64;
  repack_batch_kernel<<<(int)blocks, 256, 0, (cudaStream_t)stream>>>(jobs_device, njobs, total_units);
  WSR_LAUNCH_OK();
  return WSR_OK;
}

extern "C" int wsr_cast(const void* src, int src_dtype, void* dst, int dst_dtype, int64_t n, void* stream) {
  WSR_REQUIRE(src && dst && valid_dtype(src_dtype) && valid_dtype(dst_dtype) && n >= 0, WSR_E_INVALID, "cast: bad argument");
  if (n == 0) return WSR_OK;
  cast_kernel<<<blocks_for(n, 256), 256, 0, (cudaStream_t)stream>>>(src, src_dtype, dst, dst_dtype, n);
  WSR_LAUNCH_OK();
  return WSR_OK;
}

extern "C" int wsr_upsample2x(const void* x, int dtype, int N, int H, int W, int C, int x_ld, void* y, int y_ld, void* stream) {
  WSR_REQUIRE(x && y && valid_dtype(dtype) && N > 0 && H > 0 && W > 0 && C > 0 && x_ld >= C && y_ld >= C, WSR_E_INVALID, "upsample2x: bad argument");
  int64_t total = (int64_t)N * 4 * H * W * C;
  if (dtype == WSR_BF16) upsample2x_kernel<__nv_bfloat16><<<blocks_for(total, 256), 256, 0, (cudaStream_t)stream>>>((const __nv_bfloat16*)x, H, W, C, x_ld, (__nv_bfloat16*)y, y_ld, total);
  else upsample2x_kernel<float><<<blocks_for(total, 256), 256, 0, (cudaStream_t)stream>>>((const float*)x, H, W, C, x_ld, (float*)y, y_ld, total);
  WSR_LAUNCH_OK();
  return WSR_OK;
}

extern "C" int wsr_axpby(const void* x, int x_dtype, int x_ld, float a, const void* z, int z_dtype, int z_ld, float b,
                         void* y, int y_dtype, int y_ld, int64_t pixels, int C, void* stream) {
  WSR_REQUIRE(x && z && y && valid_dtype(x_dtype) && valid_dtype(z_dtype) && valid_dtype(y_dtype) && pixels > 0 && C > 0,
              WSR_E_INVALID, "axpby: bad argument");
  int64_t total = pixels * C;
  axpby_kernel<<<blocks_for(total, 256), 256, 0, (cudaStream_t)stream>>>(x, x_dtype, x_ld, a, z, z_dtype, z_ld, b, y, y_dtype, y_ld, C, total);
  WSR_LAUNCH_OK();
  return WSR_OK;
}

extern "C" int wsr_fill_zero(void* p, int64_t bytes, void* stream) {
  WSR_REQUIRE(p && bytes >= 0, WSR_E_INVALID, "fill_zero: bad argument");
  WSR_CUDA_OK(cudaMemsetAsync(p, 0, (size_t)bytes, (cudaStream_t)stream));
  return WSR_OK;
}

extern "C" int wsr_gn_stats(const void* x, int x_dtype, int N, int HW, int C, int x_ld, double* stats, int stats_ld, void* stream) {
  WSR_REQUIRE(x && stats && valid_dtype(x_dtype) && N > 0 && HW > 0 && C > 0 && x_ld >= C && stats_ld >= 2 * C, WSR_E_INVALID, "gn_stats: bad argument");
  GnGeom g = gn_geom(x_dtype, C, x_ld, x_ld, x, x);
  WSR_REQUIRE(g.vec != 0 && g.threads <= 1024, WSR_E_UNSUPPORTED, "gn_stats: C=%d too wide", C);
  dim3 grid((HW + g.chunk - 1) / g.chunk, N);
  size_t smem = (size_t)g.PL * C * 2 * sizeof(float);
  cudaStream_t st = (cudaStream_t)stream;
  if (x_dtype == WSR_BF16) {
    if (g.vec == 8) gn_stats_kernel<__nv_bfloat16, 8><<<grid, g.threads, smem, st>>>((const __nv_bfloat16*)x, HW, C, x_ld, g.CV, g.PL, g.chunk, stats, stats_ld);
    else gn_stats_kernel<__nv_bfloat16, 1><<<grid, g.threads, smem, st>>>((const __nv_bfloat16*)x, HW, C, x_ld, g.CV, g.PL, g.chunk, stats, stats_ld);
  } else {
    if (g.vec == 4) gn_stats_kernel<float, 4><<<grid, g.threads, smem, st>>>((const float*)x, HW, C, x_ld, g.CV, g.PL, g.chunk, stats, stats_ld);
    else gn_stats_kernel<float, 1><<<grid, g.threads, smem, st>>>((const float*)x, HW, C, x_ld, g.CV, g.PL, g.chunk, stats, stats_ld);
  }
  WSR_LAUNCH_OK();
  return WSR_OK;
}

static int gn_apply_impl(const void* x, int x_dtype, int N, int HW, int C, int x_ld, const double* stats, int stats_ld,
                         const float* gamma, const float* beta, int groups, float eps, int act, void* y, int y_dtype,
                         int y_ld, float drop_p, uint64_t drop_seed, uint32_t drop_tag, void* stream) {
  WSR_REQUIRE(x && y && stats && gamma && beta && valid_dtype(x_dtype) && N > 0 && HW > 0 && C > 0 && x_ld >= C && y_ld >= C && stats_ld >= 2 * C,
              WSR_E_INVALID, "gn_apply: bad argument");
  WSR_REQUIRE(groups > 0 && C % groups == 0, WSR_E_INVALID, "gn_apply: C=%d not divisible by groups=%d", C, groups);
  WSR_REQUIRE(y_dtype == x_dtype, WSR_E_UNSUPPORTED, "gn_apply: y_dtype must equal x_dtype");
  WSR_REQUIRE(drop_p >= 0.f && drop_p < 1.f, WSR_E_INVALID, "gn_apply: dropout p=%f", (double)drop_p);
  GnGeom g = gn_geom(x_dtype, C, x_ld, y_ld, x, y);
  WSR_REQUIRE(g.vec != 0 && g.threads <= 1024, WSR_E_UNSUPPORTED, "gn_apply: C=%d too wide", C);
  // small feature maps: shrink the per-block pixel chunk until the grid has ~4 blocks per SM
  {
    const int want = (592 + N - 1) / N;                         // blocks per image
    int chunk = (HW + want - 1) / want;
    chunk = (chunk + g.PL - 1) / g.PL * g.PL;
    if (chunk < 4 * g.PL) chunk = 4 * g.PL;
    if (chunk < g.chunk) g.chunk = chunk;
  }
  const dim3 grid((HW + g.chunk - 1) / g.chunk, N);
  size_t smem = ((size_t)C * 2 + 2 * groups) * sizeof(float);
  cudaStream_t st = (cudaStream_t)stream;
#define GN_APPLY(T, V, D) WSR_CUDA_OK(launch_pdl(gn_apply_kernel<T, T, V, D>, grid, dim3(g.threads), smem, st, (const T*)x, HW, C, x_ld, g.CV, g.PL, g.chunk, stats, stats_ld, gamma, beta, groups, eps, act, (T*)y, y_ld, drop_p, drop_seed, drop_tag))
  if (drop_p > 0.f) {
    if (x_dtype == WSR_BF16) { if (g.vec == 8) GN_APPLY(__nv_bfloat16, 8, true); else GN_APPLY(__nv_bfloat16, 1, true); }
    else { if (g.vec == 4) GN_APPLY(float, 4, true); else GN_APPLY(float, 1, true); }
  } else {
    if (x_dtype == WSR_BF16) { if (g.vec == 8) GN_APPLY(__nv_bfloat16, 8, false); else GN_APPLY(__nv_bfloat16, 1, false); }
    else { if (g.vec == 4) GN_APPLY(float, 4, false); else GN_APPLY(float, 1, false); }
  }
#undef GN_APPLY
  WSR_LAUNCH_OK();
  return WSR_OK;
}

extern "C" int wsr_gn_finalize(const double* stats, int stats_ld, int N, int HW, int C, int groups, float eps, const float* gamma,
                               const float* beta, float* table, int table_ld, void* stream) {
  WSR_REQUIRE(stats && gamma && beta && table && N > 0 && HW > 0 && C > 0 && stats_ld >= 2 * C && table_ld >= C, WSR_E_INVALID, "gn_finalize: bad argument");
  WSR_REQUIRE(groups > 0 && C % groups == 0, WSR_E_INVALID, "gn_finalize: C=%d not divisible by groups=%d", C, groups);
  gn_finalize_kernel<<<N, C >= 256 ? 256 : ((C + 31) / 32) * 32, 0, (cudaStream_t)stream>>>(stats, stats_ld, HW, C, groups, eps, gamma, beta,
                                                                                       (float2*)table, table_ld);
  WSR_LAUNCH_OK();
  return WSR_OK;
}

extern "C" int wsr_gn_apply(const void* x, int x_dtype, int N, int HW, int C, int x_ld, const double* stats, int stats_ld,
                            const float* gamma, const float* beta, int groups, float eps, int act, void* y,
                            int y_dtype, int y_ld, void* stream) {
  return gn_apply_impl(x, x_dtype, N, HW, C, x_ld, stats, stats_ld, gamma, beta, groups, eps, act, y, y_dtype, y_ld, 0.f, 0, 0, stream);
}

extern "C" int wsr_gn_apply_dropout(const void* x, int x_dtype, int N, int HW, int C, int x_ld, const double* stats,
                                    int stats_ld, const float* gamma, const float* beta, int groups, float eps, int act,
                                    void* y, int y_dtype, int y_ld, float drop_p, uint64_t drop_seed, uint32_t drop_tag,
                                    void* stream) {
  return gn_apply_impl(x, x_dtype, N, HW, C, x_ld, stats, stats_ld, gamma, beta, groups, eps, act, y, y_dtype, y_ld, drop_p, drop_seed, drop_tag, stream);
}

__global__ void dropout_mask_kernel(float* out, int64_t total, float p, uint64_t seed, uint32_t tag) {
  int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= total) return;
  float m[1];
  dropout_scale<1>(seed, tag, (uint64_t)e, p, m);
  out[e] = m[0];
}

extern "C" int wsr_dropout_mask(float* out, int N, int HW, int C, float p, uint64_t seed, uint32_t tag, void* stream) {
  WSR_REQUIRE(out && N > 0 && HW > 0 && C > 0 && p >= 0.f && p < 1.f, WSR_E_INVALID, "dropout_mask: bad argument");
  const int64_t total = (int64_t)N * HW * C;
  dropout_mask_kernel<<<blocks_for(total, 256), 256, 0, (cudaStream_t)stream>>>(out, total, p, seed, tag);
  WSR_LAUNCH_OK();
  return WSR_OK;
}

extern "C" int wsr_softmax_rows(const void* s, int s_dtype, int64_t rows, int cols, int64_t s_ld, float scale, void* p,
                                int p_dtype, int64_t p_ld, void* stream) {
  WSR_REQUIRE(s && p && valid_dtype(s_dtype) && valid_dtype(p_dtype) && rows > 0 && cols > 0 && s_ld >= cols && p_ld >= cols,
              WSR_E_INVALID, "softmax_rows: bad argument");
  WSR_REQUIRE(rows <= 2147483647LL, WSR_E_UNSUPPORTED, "softmax_rows: too many rows");
  if (s_dtype == WSR_F32 && cols % 128 == 0 && cols <= 1024 && s_ld % 4 == 0 && p_ld % 4 == 0 && (((uintptr_t)s) & 15) == 0 &&
      (((uintptr_t)p) & 15) == 0) {
    const unsigned blocks = (unsigned)((rows + 7) / 8);
    cudaStream_t st = (cudaStream_t)stream;
    const float* sf = (const float*)s;
    switch (cols / 128) {
      case 1: softmax_rows_warp_kernel<1><<<blocks, 256, 0, st>>>(sf, s_ld, scale, p, p_dtype, p_ld, rows); break;
      case 2: softmax_rows_warp_kernel<2><<<blocks, 256, 0, st>>>(sf, s_ld, scale, p, p_dtype, p_ld, rows); break;
      case 3: softmax_rows_warp_kernel<3><<<blocks, 256, 0, st>>>(sf, s_ld, scale, p, p_dtype, p_ld, rows); break;
      case 4: softmax_rows_warp_kernel<4><<<blocks, 256, 0, st>>>(sf, s_ld, scale, p, p_dtype, p_ld, rows); break;
      case 5: softmax_rows_warp_kernel<5><<<blocks, 256, 0, st>>>(sf, s_ld, scale, p, p_dtype, p_ld, rows); break;
      case 6: softmax_rows_warp_kernel<6><<<blocks, 256, 0, st>>>(sf, s_ld, scale, p, p_dtype, p_ld, rows); break;
      case 7: softmax_rows_warp_kernel<7><<<blocks, 256, 0, st>>>(sf, s_ld, scale, p, p_dtype, p_ld, rows); break;
      default: softmax_rows_warp_kernel<8><<<blocks, 256, 0, st>>>(sf, s_ld, scale, p, p_dtype, p_ld, rows); break;
    }
    WSR_LAUNCH_OK();
    return WSR_OK;
  }
  softmax_rows_kernel<<<(unsigned)rows, 128, 0, (cudaStream_t)stream>>>(s, s_dtype, cols, s_ld, scale, p, p_dtype, p_ld);
  WSR_LAUNCH_OK();
  return WSR_OK;
}

extern "C" int wsr_noise_embed(const float* level, int R, int inner, const float* w1, const float* b1, const float* w2,
                               const float* b2, int act, float* temb, void* stream) {
  WSR_REQUIRE(level && w1 && b1 && w2 && b2 && temb && R > 0 && inner > 0 && inner % 2 == 0, WSR_E_INVALID, "noise_embed: bad argument");
  WSR_REQUIRE(inner <= 2048, WSR_E_UNSUPPORTED, "noise_embed: inner=%d too large", inner);
  noise_embed_kernel<<<R, 256, (size_t)5 * inner * sizeof(float), (cudaStream_t)stream>>>(level, inner, w1, b1, w2, b2, act, temb);
  WSR_LAUNCH_OK();
  return WSR_OK;
}

extern "C" int wsr_linear_rows(const float* x, int R, int K, const float* w, const float* bias, int P, float* y, void* stream) {
  WSR_REQUIRE(x && w && y && R > 0 && K > 0 && P > 0, WSR_E_INVALID, "linear_rows: bad argument");
  WSR_REQUIRE(R <= 65535 && K <= 8192, WSR_E_UNSUPPORTED, "linear_rows: R=%d K=%d out of range", R, K);
  dim3 grid((P + 127) / 128, R);
  linear_rows_kernel<<<grid, 128, (size_t)K * sizeof(float), (cudaStream_t)stream>>>(x, K, w, bias, P, y);
  WSR_LAUNCH_OK();
  return WSR_OK;
}

extern "C" int wsr_broadcast_row(const float* table, int P, const int* row_index, int B, float* out, void* stream) {
  WSR_REQUIRE(table && row_index && out && P > 0 && B > 0 && B <= 65535, WSR_E_INVALID, "broadcast_row: bad argument");
  dim3 grid((P + 255) / 256, B);
  broadcast_row_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(table, P, row_index, out);
  WSR_LAUNCH_OK();
  return WSR_OK;
}

extern "C" int wsr_sampler_step(const float* x, const void* eps, int eps_dtype, const float* z, int64_t z_step_stride,
                                uint64_t seed, const float* tables, int T, const int* t_dev, int clip, float* x_out,
                                int64_t n, void* stream) {
  WSR_REQUIRE(x && eps && tables && t_dev && x_out && valid_dtype(eps_dtype) && T > 0 && n > 0, WSR_E_INVALID, "sampler_step: bad argument");
  sampler_step_kernel<false, false><<<blocks_for((n + 3) / 4, 256), 256, 0, (cudaStream_t)stream>>>(x, eps, eps_dtype, z, z_step_stride, seed, nullptr, 1,
                                                                                                     nullptr, tables, T, t_dev, clip, x_out, n);
  WSR_LAUNCH_OK();
  return WSR_OK;
}

extern "C" int wsr_sampler_step_members(const float* x, const void* eps, int eps_dtype, const float* z, int64_t z_step_stride,
                                        const uint64_t* member_keys, int64_t member_elems, const float* tables, int T, const int* t_dev,
                                        int clip, float* x_out, int64_t n, void* stream) {
  WSR_REQUIRE(x && eps && tables && t_dev && x_out && member_keys && valid_dtype(eps_dtype) && T > 0 && n > 0, WSR_E_INVALID,
              "sampler_step_members: bad argument");
  WSR_REQUIRE(member_elems > 0 && member_elems % 4 == 0, WSR_E_INVALID, "sampler_step_members: member_elems=%lld is not a positive multiple of 4",
              (long long)member_elems);
  sampler_step_kernel<true, false><<<blocks_for((n + 3) / 4, 256), 256, 0, (cudaStream_t)stream>>>(x, eps, eps_dtype, z, z_step_stride, 0, member_keys,
                                                                                                    member_elems / 4, nullptr, tables, T, t_dev, clip, x_out, n);
  WSR_LAUNCH_OK();
  return WSR_OK;
}

extern "C" int wsr_sampler_step_multistep(const float* x, const void* eps, int eps_dtype, float* x0_hist, const float* tables, int S,
                                          const int* t_dev, int clip, float* x_out, int64_t n, void* stream) {
  WSR_REQUIRE(x && eps && x0_hist && tables && t_dev && x_out && valid_dtype(eps_dtype) && S > 0 && n > 0, WSR_E_INVALID,
              "sampler_step_multistep: bad argument");
  sampler_step_kernel<false, true><<<blocks_for((n + 3) / 4, 256), 256, 0, (cudaStream_t)stream>>>(x, eps, eps_dtype, nullptr, 0, 0, nullptr, 1,
                                                                                                    x0_hist, tables, S, t_dev, clip, x_out, n);
  WSR_LAUNCH_OK();
  return WSR_OK;
}

extern "C" int wsr_step_counter_add(int* t_dev, int delta, void* stream) {
  WSR_REQUIRE(t_dev, WSR_E_INVALID, "step_counter_add: null");
  step_counter_add_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(t_dev, delta);
  WSR_LAUNCH_OK();
  return WSR_OK;
}

extern "C" int wsr_randn(float* out, int64_t n, uint64_t seed, uint32_t tag, void* stream) {
  WSR_REQUIRE(out && n > 0, WSR_E_INVALID, "randn: bad argument");
  randn_kernel<false><<<blocks_for((n + 3) / 4, 256), 256, 0, (cudaStream_t)stream>>>(out, n, seed, nullptr, 1, tag);
  WSR_LAUNCH_OK();
  return WSR_OK;
}

extern "C" int wsr_randn_members(float* out, int64_t n, const uint64_t* member_keys, int64_t member_elems, uint32_t tag, void* stream) {
  WSR_REQUIRE(out && member_keys && n > 0, WSR_E_INVALID, "randn_members: bad argument");
  WSR_REQUIRE(member_elems > 0 && member_elems % 4 == 0, WSR_E_INVALID, "randn_members: member_elems=%lld is not a positive multiple of 4",
              (long long)member_elems);
  randn_kernel<true><<<blocks_for((n + 3) / 4, 256), 256, 0, (cudaStream_t)stream>>>(out, n, 0, member_keys, member_elems / 4, tag);
  WSR_LAUNCH_OK();
  return WSR_OK;
}

extern "C" int wsr_q_sample(const float* hr, const float* sr, const float* noise, const float* a, int B,
                            int64_t per_sample, float* x_noisy, void* stream) {
  WSR_REQUIRE(hr && sr && noise && a && x_noisy && B > 0 && per_sample > 0, WSR_E_INVALID, "q_sample: bad argument");
  int64_t n = (int64_t)B * per_sample;
  q_sample_kernel<<<blocks_for(n, 256), 256, 0, (cudaStream_t)stream>>>(hr, sr, noise, a, per_sample, x_noisy, n);
  WSR_LAUNCH_OK();
  return WSR_OK;
}

extern "C" int wsr_noise_loss(const float* noise, const float* eps, int64_t n, int l2, double* loss, float* grad,
                              float scale, void* stream) {
  WSR_REQUIRE(noise && eps && loss && n > 0, WSR_E_INVALID, "noise_loss: bad argument");
  unsigned blocks = (unsigned)((n + 255) / 256);
  if (blocks > 1184) blocks = 1184;   // 8 CTAs per SM x 148 SMs
  noise_loss_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(noise, eps, n, l2, loss, grad, scale);
  WSR_LAUNCH_OK();
  return WSR_OK;
}
