// head.cu -- the UNet head and the reverse-step update in ONE kernel (HBM-bound):
//   eps_hat = conv3x3(Swish(GroupNorm(x)))                  final_conv, resdiff/unet.py:119,177 + nn_modules/resnet.py:19-28
//   x0 = clamp(c_recip[t] x_t - c_recipm1[t] eps_hat); x_{t-1} = coef1[t] x0 + coef2[t] x_t + sigma_t z      diffusion.py:124-125,139-141,168-169,191-192
// Round 1 ran this as three launches: gn_apply (read + write of the 64-channel full-resolution tensor), the tcgen05 convolution
// with Cout padded 1 -> 64 (11 TFLOP/s: 63 of its 64 output columns are zeros) and the sampler step.  A Cout <= 4 convolution is a
// 9 * Cin-term dot product per pixel, i.e. bandwidth-bound work: here every CTA loads a (4 + 2) x (128 + 2) pixel halo tile of the RAW
// tensor once, applies GroupNorm + Swish on the way into shared memory (bf16, 16-byte chunks XOR-swizzled by pixel so that
// neighbouring pixels hit different banks); the 9 * Cin products per pixel run on the warp-level tensor path (mma.sync m16n8k16, bf16
// operands fetched with ldmatrix from the swizzled tile, the <= 4 output channels padded to n = 8, fp32 accumulation) -- a CUDA-core
// version of the same loop issued 5x the instructions and was bound by them (0.34 ms at batch 64) -- and the epilogue is the sampler
// update, in place on the fp32 NCHW state.  tcgen05 is the wrong tool here: its smallest tile (M = 128, N = 16) leaves the kernel
// bound by the activation-operand fetch exactly as the Cout-padded convolution was.  Algorithmic traffic: Cin * 2 bytes per pixel
// read (+ halo) and 12-16 bytes per pixel-channel for the state update.
#include "common.cuh"
#include "philox.cuh"

namespace wsr {

constexpr int kHeadRows = 4, kHeadCols = 128, kHeadThreads = 256;
constexpr int kHeadMaxCout = 4;

struct HeadParams {
  const __nv_bfloat16* x; int x_ld;       // raw (pre-GroupNorm) input, NHWC (B, H, W, Cin) bf16
  int B, H, W, Cin, Cout;
  const double* stats; int stats_ld; const float* gamma; const float* beta; int groups; float gn_eps;
  const uint4* w;                          // bf16, ldmatrix-ready blocks (wsr_pack_head_weight), (Cin / 64) * 9 * 4 * 2 * 128 bytes
  const float* bias;                       // [Cout] or null
  float* eps_out;                          // fp32 NCHW (B, Cout, H, W) or null
  float* xs;                               // fp32 NCHW state x_t -> x_{t-1} in place, or null (convolution only)
  const float* z; long long z_stride; unsigned long long seed; const float* tab; int T; const int* t_dev; int clip;
  const unsigned long long* member_keys; long long member_groups;   // ensemble batch (MK): per-member Philox keys, member elements / 4
  float* hist;                             // multistep (MS): fp32 NCHW x0 of the previous step, read when c_prev != 0, then overwritten
};

__device__ __forceinline__ void head_randn4(uint64_t seed, uint32_t tag, uint64_t grp, float (&z)[4]) {
  // identical stream layout to randn4 of elementwise.cu (wsr_sampler_step / wsr_randn): element i = word i & 3 of group i >> 2
  uint32_t c[4] = {(uint32_t)grp, (uint32_t)(grp >> 32), tag, 0x5752u};
  philox4x32_10(c, (uint32_t)seed, (uint32_t)(seed >> 32));
  const float s = 2.3283064365386963e-10f;
  float u0 = ((float)c[0] + 0.5f) * s, u1 = ((float)c[1] + 0.5f) * s;
  float u2 = ((float)c[2] + 0.5f) * s, u3 = ((float)c[3] + 0.5f) * s;
  float r0 = sqrtf(-2.f * __logf(u0)), r1 = sqrtf(-2.f * __logf(u2));
  float s0, c0, s1, c1;
  __sincosf(6.283185307179586f * u1, &s0, &c0);
  __sincosf(6.283185307179586f * u3, &s1, &c1);
  z[0] = r0 * c0; z[1] = r0 * s0; z[2] = r1 * c1; z[3] = r1 * s1;
}

// shared memory: tile [Cin/64 planes][6 rows][130 cols][64 ch] bf16 | weights bf16 as ldmatrix-ready 8x8 blocks
// [plane][tap][16-channel step][k half][n = 8 output channels (zero above Cout)][8 channels] | scale[Cin] shift[Cin] | group moments
// MS: the epilogue is the multistep update of wsr_sampler_step_multistep (tables (c_recip, c_recipm1, c_x0, c_x, c_prev), no noise)
template <int COUT, bool MK, bool MS>
__global__ void __launch_bounds__(kHeadThreads) head_sampler_kernel(const HeadParams p) {
  extern __shared__ __align__(16) uint8_t hsm[];
  constexpr int TR = kHeadRows + 2, TC = kHeadCols + 2;
  const int planes = p.Cin >> 6;
  uint8_t* tile = hsm;
  __nv_bfloat16* wsm = (__nv_bfloat16*)(hsm + (size_t)planes * TR * TC * 128);
  float* sc = (float*)(wsm + (size_t)planes * 9 * 4 * 2 * 64);
  float* sh = sc + p.Cin;
  float* gm = sh + p.Cin;
  const int n = blockIdx.y;
  const int tiles_x = (p.W + kHeadCols - 1) / kHeadCols;
  const int ty = blockIdx.x / tiles_x, tx = blockIdx.x - ty * tiles_x;
  const int y0 = ty * kHeadRows, x0 = tx * kHeadCols;
  const int tid = threadIdx.x;

  // ---- halo tile loader: raw bf16 -> GroupNorm + Swish -> bf16 (out-of-image pixels = the convolution's zero padding).  The global
  // loads are issued kU at a time BEFORE their results are needed (a block is one latency chain otherwise: 25 dependent ~1 us round
  // trips per thread), and the first batch is in flight while the weights / GroupNorm parameters are staged.
  constexpr int kU = 7;
  const int nvec = planes * TR * TC * 8;                 // 16-byte vectors (8 channels)
  const __nv_bfloat16* xb = p.x + (long long)n * p.H * p.W * p.x_ld;
  uint4 raw[kU];
  auto locate = [&](int v, int& k, int& col, int& row, int& pl) -> bool {
    k = v & 7;
    int r = v >> 3;
    col = r % TC; r /= TC;
    row = r % TR; pl = r / TR;
    const int gy = y0 + row - 1, gx = x0 + col - 1;
    return v < nvec && gy >= 0 && gy < p.H && gx >= 0 && gx < p.W;
  };
  auto issue = [&](int v0) {
#pragma unroll
    for (int u = 0; u < kU; ++u) {
      int k, col, row, pl;
      raw[u] = make_uint4(0u, 0u, 0u, 0u);
      if (locate(v0 + u * kHeadThreads, k, col, row, pl))
        raw[u] = __ldg((const uint4*)(xb + ((long long)(y0 + row - 1) * p.W + (x0 + col - 1)) * p.x_ld + pl * 64 + k * 8));
    }
  };
  pdl_launch_dependents();
  pdl_wait();
  issue(tid);
  for (int i = tid; i < planes * 9 * 4 * 2 * 8; i += kHeadThreads) ((uint4*)wsm)[i] = __ldg(p.w + i);
  {
    const int cpg = p.Cin / p.groups;
    const long long HW = (long long)p.H * p.W;
    for (int g = tid; g < p.groups; g += kHeadThreads) {
      double a = 0.0, b = 0.0;
      for (int j = 0; j < cpg; ++j) { a += p.stats[(long long)n * p.stats_ld + (g * cpg + j) * 2]; b += p.stats[(long long)n * p.stats_ld + (g * cpg + j) * 2 + 1]; }
      const double inv_cnt = 1.0 / ((double)cpg * (double)HW);
      const double mean = a * inv_cnt;
      double var = b * inv_cnt - mean * mean;
      if (var < 0.0) var = 0.0;
      gm[2 * g] = (float)mean;
      gm[2 * g + 1] = rsqrtf((float)var + p.gn_eps);
    }
    __syncthreads();
    for (int c = tid; c < p.Cin; c += kHeadThreads) {
      const int g = c / cpg;
      const float s = p.gamma[c] * gm[2 * g + 1];
      sc[c] = s;
      sh[c] = p.beta[c] - gm[2 * g] * s;
    }
    __syncthreads();
  }
  for (int v0 = tid; v0 < nvec; v0 += kU * kHeadThreads) {
    uint4 cur[kU];
#pragma unroll
    for (int u = 0; u < kU; ++u) cur[u] = raw[u];
    if (v0 + kU * kHeadThreads < nvec) issue(v0 + kU * kHeadThreads);          // next batch in flight while this one is transformed
#pragma unroll
    for (int u = 0; u < kU; ++u) {
      int k, col, row, pl;
      const int v = v0 + u * kHeadThreads;
      const bool inside = locate(v, k, col, row, pl);
      if (v >= nvec) continue;
      uint4 o = make_uint4(0u, 0u, 0u, 0u);
      if (inside) {
        const int c0 = pl * 64 + k * 8;
        const __nv_bfloat162* h = (const __nv_bfloat162*)&cur[u];
        __nv_bfloat162* oh = (__nv_bfloat162*)&o;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const float2 f = __bfloat1622float2(h[q]);
          const float a0 = swish_fast(fmaf(f.x, sc[c0 + 2 * q], sh[c0 + 2 * q]));
          const float a1 = swish_fast(fmaf(f.y, sc[c0 + 2 * q + 1], sh[c0 + 2 * q + 1]));
          oh[q] = __floats2bfloat162_rn(a0, a1);
        }
      }
      *(uint4*)(tile + ((size_t)(pl * TR + row) * TC + col) * 128 + ((k ^ (col & 7)) << 4)) = o;
    }
  }
  __syncthreads();
  // ---- 9 * Cin products per pixel on mma.sync m16n8k16: warp w owns row w >> 1, columns (w & 1) * 64 .. + 63 = four 16-pixel M tiles ----
  const int warp = tid >> 5, lane = tid & 31;
  const int r = warp >> 1, cbase = (warp & 1) * 64;
  float acc[4][4];
#pragma unroll
  for (int mt = 0; mt < 4; ++mt)
#pragma unroll
    for (int q = 0; q < 4; ++q) acc[mt][q] = 0.f;
  const uint32_t tile_s = (uint32_t)__cvta_generic_to_shared(tile);
  const uint32_t wsm_s = (uint32_t)__cvta_generic_to_shared(wsm);
  // ldmatrix row addresses: A -- lane l supplies pixel (l & 7) + 8 * ((l >> 3) & 1) of the M tile, k half l >> 4;
  //                         B -- lanes 0..15 supply row (l & 7) of k-half matrix (l >> 3) & 1
  const int a_px = (lane & 7) + ((lane >> 3) & 1) * 8, a_kh = lane >> 4;
  const uint32_t b_off = (uint32_t)((((lane >> 3) & 1) * 8 + (lane & 7)) * 16);
  for (int pl = 0; pl < planes; ++pl) {
#pragma unroll 1
    for (int tap = 0; tap < 9; ++tap) {
      const int dy = tap / 3, dx = tap - dy * 3;
      const uint32_t rowp = tile_s + (uint32_t)(((pl * TR + r + dy) * TC) * 128);
#pragma unroll
      for (int kc = 0; kc < 4; ++kc) {
        uint32_t b0, b1;
        asm volatile("ldmatrix.sync.aligned.m8n8.x2.shared.b16 {%0, %1}, [%2];" : "=r"(b0), "=r"(b1)
                     : "r"(wsm_s + (uint32_t)((((pl * 9 + tap) * 4 + kc) * 2) * 128) + b_off));
        const int chunk = kc * 2 + a_kh;
#pragma unroll
        for (int mt = 0; mt < 4; ++mt) {
          const int col = cbase + mt * 16 + a_px + dx;
          uint32_t a0, a1, a2, a3;
          asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0, %1, %2, %3}, [%4];" : "=r"(a0), "=r"(a1), "=r"(a2), "=r"(a3)
                       : "r"(rowp + (uint32_t)(col * 128 + ((chunk ^ (col & 7)) << 4))));
          asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
                       : "+f"(acc[mt][0]), "+f"(acc[mt][1]), "+f"(acc[mt][2]), "+f"(acc[mt][3]) : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
        }
      }
    }
  }
  // accumulator (m16n8): lane l holds pixels l >> 2 (c0, c1) and (l >> 2) + 8 (c2, c3) of each M tile for output channels 2 (l & 3), + 1.
  // Re-distribute so that lane l owns pixels l and l + 32 of the warp's 64 (all output channels): pixel P = mt * 16 + q sits in
  // lane (q & 7) * 4 + (co >> 1), register (q >> 3) * 2 + (co & 1) of M tile mt.
  float outv[2][COUT];
  {
    const int q = lane & 15, want_hi = q >> 3, want_mt = lane >> 4;
#pragma unroll
    for (int co = 0; co < COUT; ++co) {
      const int src = (q & 7) * 4 + (co >> 1);
#pragma unroll
      for (int px = 0; px < 2; ++px) {
        float v = 0.f;
#pragma unroll
        for (int m2 = 0; m2 < 2; ++m2)
#pragma unroll
          for (int hi = 0; hi < 2; ++hi) {
            const float cand = __shfl_sync(0xffffffffu, acc[px * 2 + m2][hi * 2 + (co & 1)], src);
            if (m2 == want_mt && hi == want_hi) v = cand;
          }
        outv[px][co] = v + (p.bias ? p.bias[co] : 0.f);
      }
    }
  }
  const int j = cbase + lane;                      // tile column of this lane's first pixel; the second one is j + 32
  // ---- epilogue: eps_hat (optional) and the reverse-step update of the state, fp32 NCHW ----
  const int gy = y0 + r;
  if (gy >= p.H) return;
  int t = 0;
  float c_recip = 0.f, c_recipm1 = 0.f, coef1 = 0.f, coef2 = 0.f, sigma = 0.f;
  const float* zt = nullptr;
  float c_prev = 0.f;
  if (p.xs) {
    t = *p.t_dev;
    c_recip = p.tab[t]; c_recipm1 = p.tab[p.T + t]; coef1 = p.tab[2 * p.T + t]; coef2 = p.tab[3 * p.T + t];
    if constexpr (MS) {
      c_prev = p.tab[4 * p.T + t];
    } else {
      sigma = t > 0 ? __expf(0.5f * p.tab[4 * p.T + t]) : 0.f;
      if (p.z) zt = p.z + (long long)(p.T - t) * p.z_stride;
    }
  }
#pragma unroll
  for (int px = 0; px < 2; ++px) {
    const int gx = x0 + j + 32 * px;
    if (gx >= p.W) continue;
#pragma unroll
    for (int co = 0; co < COUT; ++co) {
      const long long i = (((long long)n * COUT + co) * p.H + gy) * p.W + gx;
      const float e = outv[px][co];
      if (p.eps_out) p.eps_out[i] = e;
      if (MS && p.xs) {
        const float xv = p.xs[i];
        float x0v = c_recip * xv - c_recipm1 * e;
        if (p.clip) x0v = fminf(1.f, fmaxf(-1.f, x0v));
        float o = coef1 * x0v + coef2 * xv;
        if (c_prev != 0.f) o += c_prev * p.hist[i];
        p.hist[i] = x0v;
        p.xs[i] = o;
      } else if (p.xs) {
        float zz = 0.f;
        if (t > 0) {
          if (zt) zz = zt[i];
          else {
            // MK: member m = group / member_groups draws from its own key at the member-local group (wsr_sampler_step_members)
            long long grp = i >> 2;
            unsigned long long key = p.seed;
            if constexpr (MK) {
              const long long m = grp / p.member_groups;
              grp -= m * p.member_groups;
              key = __ldg(p.member_keys + m);
            }
            float z4[4]; head_randn4(key, (uint32_t)t, (uint64_t)grp, z4); const int wsel = (int)(i & 3); zz = wsel == 0 ? z4[0] : wsel == 1 ? z4[1] : wsel == 2 ? z4[2] : z4[3];
          }
        }
        const float xv = p.xs[i];
        float x0v = c_recip * xv - c_recipm1 * e;
        if (p.clip) x0v = fminf(1.f, fmaxf(-1.f, x0v));
        p.xs[i] = coef1 * x0v + coef2 * xv + sigma * zz;
      }
    }
  }
}

// fp32 [9][Cout][Cin] (wsr_pack_conv_weight layout) -> bf16 blocks [plane][tap][16-channel step][k half][n = 8][8 channels], rows n >= Cout zero
__global__ void pack_head_weight_kernel(const float* __restrict__ w, int Cout, int Cin, __nv_bfloat16* __restrict__ dst, int total) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int kk = i & 7, nn = (i >> 3) & 7, h = (i >> 6) & 1, kc = (i >> 7) & 3;
  const int tp = i >> 9, tap = tp % 9, pl = tp / 9;
  dst[i] = __float2bfloat16_rn(nn < Cout ? w[((long long)tap * Cout + nn) * Cin + pl * 64 + kc * 16 + h * 8 + kk] : 0.f);
}

static size_t head_smem_bytes(int Cin, int Cout, int groups) {
  (void)Cout;
  return (size_t)(Cin / 64) * (kHeadRows + 2) * (kHeadCols + 2) * 128 + (size_t)(Cin / 64) * 9 * 4 * 2 * 128 + (size_t)(2 * Cin + 2 * groups) * 4;
}

template <int COUT, bool MK, bool MS>
static int launch_head(const HeadParams& p, cudaStream_t st) {
  const size_t smem = head_smem_bytes(p.Cin, COUT, p.groups);
  static size_t attr = 0;
  if (smem > attr) {
    WSR_CUDA_OK(cudaFuncSetAttribute(head_sampler_kernel<COUT, MK, MS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr = smem;
  }
  const int tiles = ((p.W + kHeadCols - 1) / kHeadCols) * ((p.H + kHeadRows - 1) / kHeadRows);
  WSR_CUDA_OK(launch_pdl(head_sampler_kernel<COUT, MK, MS>, dim3(tiles, p.B), dim3(kHeadThreads), smem, st, p));
  return WSR_OK;
}

}  // namespace wsr

using namespace wsr;

extern "C" int wsr_head_sampler_supported(int Cin, int Cout, int groups) {
  if (Cin <= 0 || Cin % 64 != 0 || Cout < 1 || Cout > kHeadMaxCout || groups <= 0 || Cin % groups != 0) return 0;
  return head_smem_bytes(Cin, Cout, groups) <= 227 * 1024 ? 1 : 0;
}

extern "C" int wsr_pack_head_weight(const float* w, int Cout, int Cin, void* dst, void* stream) {
  WSR_REQUIRE(w && dst && Cout >= 1 && Cout <= kHeadMaxCout && Cin > 0 && Cin % 64 == 0, WSR_E_INVALID, "pack_head_weight: bad argument");
  const int total = (Cin / 64) * 9 * 4 * 2 * 64;
  pack_head_weight_kernel<<<(total + 255) / 256, 256, 0, (cudaStream_t)stream>>>(w, Cout, Cin, (__nv_bfloat16*)dst, total);
  WSR_LAUNCH_OK();
  return WSR_OK;
}

static int head_sampler_step(const void* x, int x_ld, int B, int H, int W, int Cin, const double* stats, int stats_ld,
                             const float* gamma, const float* beta, int groups, float gn_eps, const void* w, const float* bias, int Cout,
                             float* eps_out, float* x_state, const float* z, int64_t z_step_stride, uint64_t seed,
                             const uint64_t* member_keys, int64_t member_elems, float* hist, const float* tables, int T, const int* t_dev,
                             int clip, void* stream) {
  WSR_REQUIRE(x && stats && gamma && beta && w, WSR_E_INVALID, "final_conv_sampler_step: null pointer");
  WSR_REQUIRE(B > 0 && B <= 65535 && H > 0 && W > 0, WSR_E_INVALID, "final_conv_sampler_step: bad shape");
  WSR_REQUIRE(wsr_head_sampler_supported(Cin, Cout, groups), WSR_E_UNSUPPORTED,
              "final_conv_sampler_step: needs Cin %% 64 == 0, 1 <= Cout <= 4, Cin %% groups == 0 and the tile in shared memory (Cin=%d Cout=%d)", Cin, Cout);
  WSR_REQUIRE(x_ld % 8 == 0 && x_ld >= Cin && (((uintptr_t)x) & 15) == 0 && (((uintptr_t)w) & 15) == 0, WSR_E_UNSUPPORTED,
              "final_conv_sampler_step: pitch / alignment");
  WSR_REQUIRE(eps_out || x_state, WSR_E_INVALID, "final_conv_sampler_step: no output");
  WSR_REQUIRE(!x_state || (tables && t_dev && T > 0), WSR_E_INVALID, "final_conv_sampler_step: sampler tables");
  HeadParams p;
  p.x = (const __nv_bfloat16*)x; p.x_ld = x_ld; p.B = B; p.H = H; p.W = W; p.Cin = Cin; p.Cout = Cout;
  p.stats = stats; p.stats_ld = stats_ld; p.gamma = gamma; p.beta = beta; p.groups = groups; p.gn_eps = gn_eps;
  p.w = (const uint4*)w; p.bias = bias; p.eps_out = eps_out; p.xs = x_state; p.z = z; p.z_stride = z_step_stride; p.seed = seed;
  p.tab = tables; p.T = T; p.t_dev = t_dev; p.clip = clip;
  p.member_keys = (const unsigned long long*)member_keys; p.member_groups = member_elems / 4; p.hist = hist;
  cudaStream_t st = (cudaStream_t)stream;
  if (hist) {
    switch (Cout) {
      case 1: return launch_head<1, false, true>(p, st);
      case 2: return launch_head<2, false, true>(p, st);
      case 3: return launch_head<3, false, true>(p, st);
      default: return launch_head<4, false, true>(p, st);
    }
  }
  if (member_keys) {
    switch (Cout) {
      case 1: return launch_head<1, true, false>(p, st);
      case 2: return launch_head<2, true, false>(p, st);
      case 3: return launch_head<3, true, false>(p, st);
      default: return launch_head<4, true, false>(p, st);
    }
  }
  switch (Cout) {
    case 1: return launch_head<1, false, false>(p, st);
    case 2: return launch_head<2, false, false>(p, st);
    case 3: return launch_head<3, false, false>(p, st);
    default: return launch_head<4, false, false>(p, st);
  }
}

extern "C" int wsr_final_conv_sampler_step(const void* x, int x_ld, int B, int H, int W, int Cin, const double* stats, int stats_ld,
                                           const float* gamma, const float* beta, int groups, float gn_eps, const void* w,
                                           const float* bias, int Cout, float* eps_out, float* x_state, const float* z,
                                           int64_t z_step_stride, uint64_t seed, const float* tables, int T, const int* t_dev,
                                           int clip, void* stream) {
  return head_sampler_step(x, x_ld, B, H, W, Cin, stats, stats_ld, gamma, beta, groups, gn_eps, w, bias, Cout, eps_out, x_state, z,
                           z_step_stride, seed, nullptr, 0, nullptr, tables, T, t_dev, clip, stream);
}

extern "C" int wsr_final_conv_sampler_step_members(const void* x, int x_ld, int B, int H, int W, int Cin, const double* stats,
                                                   int stats_ld, const float* gamma, const float* beta, int groups, float gn_eps,
                                                   const void* w, const float* bias, int Cout, float* eps_out, float* x_state,
                                                   const float* z, int64_t z_step_stride, const uint64_t* member_keys,
                                                   int64_t member_elems, const float* tables, int T, const int* t_dev, int clip,
                                                   void* stream) {
  WSR_REQUIRE(member_keys, WSR_E_INVALID, "final_conv_sampler_step_members: null member_keys");
  WSR_REQUIRE(member_elems > 0 && member_elems % 4 == 0, WSR_E_INVALID,
              "final_conv_sampler_step_members: member_elems=%lld is not a positive multiple of 4", (long long)member_elems);
  return head_sampler_step(x, x_ld, B, H, W, Cin, stats, stats_ld, gamma, beta, groups, gn_eps, w, bias, Cout, eps_out, x_state, z,
                           z_step_stride, 0, member_keys, member_elems, nullptr, tables, T, t_dev, clip, stream);
}

extern "C" int wsr_final_conv_sampler_step_multistep(const void* x, int x_ld, int B, int H, int W, int Cin, const double* stats,
                                                     int stats_ld, const float* gamma, const float* beta, int groups, float gn_eps,
                                                     const void* w, const float* bias, int Cout, float* eps_out, float* x_state,
                                                     float* x0_hist, const float* tables, int S, const int* t_dev, int clip, void* stream) {
  WSR_REQUIRE(x_state && x0_hist && tables, WSR_E_INVALID, "final_conv_sampler_step_multistep: null state, history or tables");
  return head_sampler_step(x, x_ld, B, H, W, Cin, stats, stats_ld, gamma, beta, groups, gn_eps, w, bias, Cout, eps_out, x_state, nullptr,
                           0, 0, nullptr, 0, x0_hist, tables, S, t_dev, clip, stream);
}
