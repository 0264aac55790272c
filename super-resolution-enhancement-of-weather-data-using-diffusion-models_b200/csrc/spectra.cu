// spectra.cu -- zonal power spectra and row error sums of output fields (wsr_zonal_spectra), the accumulators behind
// training.metrics.FieldScores.  One CTA owns one (plane, row): it stages the row(s) and a double twiddle table in shared memory
// and its threads stride over the wavenumbers k = 0 .. W/2, each summing its DFT bins directly in double over the W longitudes.
// A direct DFT keeps the high-wavenumber bins of smooth fields exact (no butterfly rounding), as the condition branch of fd.cu
// does; the cost (~2.2 GFLOP fp64 for 64 fields of 128x256) is small against the sampling that produced the fields.  Every
// accumulator slot belongs to one CTA, so the kernel needs no atomics and repeated calls are bit-identical.
#include "common.cuh"

namespace wsr {

constexpr int kSpecBlock = 128;
constexpr int kSpecMaxW = 2048;

// smem: tw[W] (double2, exp(-2 pi i n / W)), p[W], t[W] (fp32 rows as given; scale and shift are applied to the DFT sums)
template <bool HAS_T>
__global__ void __launch_bounds__(kSpecBlock) zonal_spectra_kernel(const float* __restrict__ pred, const float* __restrict__ target, int H,
                                                                   int W, const float* __restrict__ scale, const float* __restrict__ shift,
                                                                   double* __restrict__ acc) {
  extern __shared__ double2 tw[];
  float* sp = reinterpret_cast<float*>(tw + W);
  float* st = sp + W;
  __shared__ double red[kSpecBlock / 32][3];
  const int64_t row = blockIdx.x;
  const int plane = (int)(row / H);
  const int tid = threadIdx.x;
  const int K = W / 2, nb = K + 1;
  for (int n = tid; n < W; n += kSpecBlock) {
    double s, c;
    sincospi(-2.0 * (double)n / (double)W, &s, &c);
    tw[n] = make_double2(c, s);
    sp[n] = pred[row * W + n];
    if (HAS_T) st[n] = target[row * W + n];
  }
  __syncthreads();
  const double sc = scale ? (double)scale[plane] : 1.0;
  const double sh = shift ? (double)shift[plane] : 0.0;
  const double inv_w2 = 1.0 / ((double)W * (double)W);
  double* out = acc + row * (int64_t)(3 * nb + 3);
  for (int k = tid; k <= K; k += kSpecBlock) {
    double pr = 0.0, pi = 0.0, tr = 0.0, ti = 0.0, er = 0.0, ei = 0.0;
    int idx = 0;
    for (int n = 0; n < W; ++n) {
      const double2 w = tw[idx];
      const double a = (double)sp[n];
      pr = fma(a, w.x, pr);
      pi = fma(a, w.y, pi);
      if (HAS_T) {
        const double b = (double)st[n], d = a - b;      // exact: the difference of two floats fits a double
        tr = fma(b, w.x, tr);
        ti = fma(b, w.y, ti);
        er = fma(d, w.x, er);
        ei = fma(d, w.y, ei);
      }
      idx += k;
      if (idx >= W) idx -= W;
    }
    // the shift only moves the mean (k = 0); it cancels in the error
    const double c = (k == 0 || k == K) ? inv_w2 : 2.0 * inv_w2;
    const double ofs = k == 0 ? (double)W * sh : 0.0;
    const double xr = fma(sc, pr, ofs), xi = sc * pi;
    out[k] += c * (xr * xr + xi * xi);
    if (HAS_T) {
      const double yr = fma(sc, tr, ofs), yi = sc * ti, dr = sc * er, di = sc * ei;
      out[nb + k] += c * (yr * yr + yi * yi);
      out[2 * nb + k] += c * (dr * dr + di * di);
    }
  }
  if (!HAS_T) return;
  double s_abs = 0.0, s_sq = 0.0, s_d = 0.0;
  for (int n = tid; n < W; n += kSpecBlock) {
    const double d = sc * ((double)sp[n] - (double)st[n]);
    s_abs += fabs(d);
    s_sq = fma(d, d, s_sq);
    s_d += d;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    s_abs += __shfl_xor_sync(0xffffffffu, s_abs, o);
    s_sq += __shfl_xor_sync(0xffffffffu, s_sq, o);
    s_d += __shfl_xor_sync(0xffffffffu, s_d, o);
  }
  const int warp = tid >> 5;
  if ((tid & 31) == 0) { red[warp][0] = s_abs; red[warp][1] = s_sq; red[warp][2] = s_d; }
  __syncthreads();
  if (tid < 3) {
    double v = 0.0;
    for (int w = 0; w < kSpecBlock / 32; ++w) v += red[w][tid];
    out[3 * nb + tid] += v;
  }
}

}  // namespace wsr

using namespace wsr;

extern "C" int wsr_zonal_spectra(const float* pred, const float* target, int planes, int H, int W, const float* scale, const float* shift,
                                 double* acc, void* stream) {
  WSR_REQUIRE(pred && acc && planes > 0 && H > 0, WSR_E_INVALID, "zonal_spectra: bad argument");
  WSR_REQUIRE(W >= 4 && W <= kSpecMaxW && W % 2 == 0, WSR_E_UNSUPPORTED, "zonal_spectra: W=%d is not even in 4..%d", W, kSpecMaxW);
  const int64_t rows = (int64_t)planes * H;
  WSR_REQUIRE(rows <= 0x7fffffff, WSR_E_UNSUPPORTED, "zonal_spectra: planes * H = %lld rows", (long long)rows);
  const size_t smem = (size_t)W * (sizeof(double2) + 2 * sizeof(float));
  static bool attr = false;
  if (!attr) {
    const int max_smem = (int)((size_t)kSpecMaxW * (sizeof(double2) + 2 * sizeof(float)));
    WSR_CUDA_OK(cudaFuncSetAttribute(zonal_spectra_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem));
    WSR_CUDA_OK(cudaFuncSetAttribute(zonal_spectra_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem));
    attr = true;
  }
  cudaStream_t st = (cudaStream_t)stream;
  if (target)
    zonal_spectra_kernel<true><<<(unsigned)rows, kSpecBlock, smem, st>>>(pred, target, H, W, scale, shift, acc);
  else
    zonal_spectra_kernel<false><<<(unsigned)rows, kSpecBlock, smem, st>>>(pred, nullptr, H, W, scale, shift, acc);
  WSR_LAUNCH_OK();
  return WSR_OK;
}
