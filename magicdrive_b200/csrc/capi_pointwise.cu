// Memory-bound helpers of the denoising step: residual add, nearest resize, layout / dtype conversion,
// sinusoidal + Fourier embeddings, the skinny linear layers, the tiny-channel direct convolution and the fused
// classifier-free-guidance + DDIM update.  Compiled WITHOUT --use_fast_math (sin/cos/exp/erf are exact-path).
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <math.h>

#include "../../include/magicdrive_b200.h"
#include "common_host.h"

namespace {

__global__ void add_kernel(const uint4* __restrict__ a, const uint4* __restrict__ b, uint4* __restrict__ o, long long n8) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n8) return;
  const uint4 ua = __ldg(a + i), ub = __ldg(b + i);
  const __nv_bfloat162* ha = reinterpret_cast<const __nv_bfloat162*>(&ua);
  const __nv_bfloat162* hb = reinterpret_cast<const __nv_bfloat162*>(&ub);
  uint4 r;
  __nv_bfloat162* hr = reinterpret_cast<__nv_bfloat162*>(&r);
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const float2 fa = __bfloat1622float2(ha[j]), fb = __bfloat1622float2(hb[j]);
    hr[j] = __floats2bfloat162_rn(fa.x + fb.x, fa.y + fb.y);
  }
  o[i] = r;
}

__global__ void upsample_nearest_kernel(const uint4* __restrict__ x, int n, int h, int w, int c8, uint4* __restrict__ o,
                                        int ho, int wo) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  const long long total = static_cast<long long>(n) * ho * wo * c8;
  if (i >= total) return;
  const int cv = static_cast<int>(i % c8);
  long long p = i / c8;
  const int ow = static_cast<int>(p % wo);
  p /= wo;
  const int oh = static_cast<int>(p % ho);
  const int img = static_cast<int>(p / ho);
  // ATen nearest: src = min(floor(dst * (in / out)), in - 1) with the scale computed in float
  const float sh = static_cast<float>(h) / static_cast<float>(ho), sw = static_cast<float>(w) / static_cast<float>(wo);
  const int ih = min(static_cast<int>(floorf(oh * sh)), h - 1);
  const int iw = min(static_cast<int>(floorf(ow * sw)), w - 1);
  o[i] = __ldg(x + ((static_cast<long long>(img) * h + ih) * w + iw) * c8 + cv);
}

// AdaptiveAvgPool2d over NHWC fp32 (+ optional SiLU): window [floor(o * in / out), ceil((o + 1) * in / out)) like ATen
__global__ void adaptive_avgpool_kernel(const float* __restrict__ x, int n, int h, int w, int c, float* __restrict__ o, int ho,
                                        int wo, int silu) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  const long long total = static_cast<long long>(n) * ho * wo * c;
  if (i >= total) return;
  const int ch = static_cast<int>(i % c);
  long long p = i / c;
  const int ow = static_cast<int>(p % wo);
  p /= wo;
  const int oh = static_cast<int>(p % ho);
  const int img = static_cast<int>(p / ho);
  const int h0 = (oh * h) / ho, h1 = ((oh + 1) * h + ho - 1) / ho;
  const int w0 = (ow * w) / wo, w1 = ((ow + 1) * w + wo - 1) / wo;
  float acc = 0.f;
  for (int ih = h0; ih < h1; ++ih)
    for (int iw = w0; iw < w1; ++iw) acc += __ldg(x + ((static_cast<long long>(img) * h + ih) * w + iw) * c + ch);
  acc /= static_cast<float>((h1 - h0) * (w1 - w0));
  o[i] = silu ? acc / (1.0f + expf(-acc)) : acc;
}

template <typename T>
__device__ __forceinline__ float ldf(const T* p);
template <>
__device__ __forceinline__ float ldf<float>(const float* p) { return *p; }
template <>
__device__ __forceinline__ float ldf<__nv_bfloat16>(const __nv_bfloat16* p) { return __bfloat162float(*p); }

// NCHW -> NHWC through a 32x32 smem transpose tile over (c, hw)
template <typename T>
__global__ void nchw_to_nhwc_kernel(const T* __restrict__ x, int c, int hw, __nv_bfloat16* __restrict__ o) {
  __shared__ float tile[32][33];
  const int img = blockIdx.z;
  const int c0 = blockIdx.y * 32, p0 = blockIdx.x * 32;
  for (int j = threadIdx.y; j < 32; j += blockDim.y) {
    const int cc = c0 + j, p = p0 + threadIdx.x;
    if (cc < c && p < hw) tile[j][threadIdx.x] = ldf(x + (static_cast<long long>(img) * c + cc) * hw + p);
  }
  __syncthreads();
  for (int j = threadIdx.y; j < 32; j += blockDim.y) {
    const int p = p0 + j, cc = c0 + threadIdx.x;
    if (cc < c && p < hw) o[(static_cast<long long>(img) * hw + p) * c + cc] = __float2bfloat16_rn(tile[threadIdx.x][j]);
  }
}
template <typename T>
__device__ __forceinline__ void stf(T* p, float v);
template <>
__device__ __forceinline__ void stf<float>(float* p, float v) { *p = v; }
template <>
__device__ __forceinline__ void stf<__nv_bfloat16>(__nv_bfloat16* p, float v) { *p = __float2bfloat16_rn(v); }
template <typename T>
__global__ void nhwc_to_nchw_kernel(const __nv_bfloat16* __restrict__ x, int c, int hw, T* __restrict__ o) {
  __shared__ float tile[32][33];
  const int img = blockIdx.z;
  const int c0 = blockIdx.y * 32, p0 = blockIdx.x * 32;
  for (int j = threadIdx.y; j < 32; j += blockDim.y) {
    const int p = p0 + j, cc = c0 + threadIdx.x;
    if (cc < c && p < hw) tile[j][threadIdx.x] = __bfloat162float(x[(static_cast<long long>(img) * hw + p) * c + cc]);
  }
  __syncthreads();
  for (int j = threadIdx.y; j < 32; j += blockDim.y) {
    const int cc = c0 + j, p = p0 + threadIdx.x;
    if (cc < c && p < hw) stf(o + (static_cast<long long>(img) * c + cc) * hw + p, tile[threadIdx.x][j]);
  }
}

__global__ void f32_to_bf16_kernel(const float* __restrict__ x, __nv_bfloat16* __restrict__ o, long long n) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i < n) o[i] = __float2bfloat16_rn(x[i]);
}
__global__ void bf16_to_f32_kernel(const __nv_bfloat16* __restrict__ x, float* __restrict__ o, long long n) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i < n) o[i] = __bfloat162float(x[i]);
}

// get_timestep_embedding (embeddings.py:24-64): emb = t * exp(-ln(10000) * i / (half - shift)); [sin | cos], flipped.
__global__ void timestep_embedding_kernel(const float* __restrict__ t, int m, int dim, int flip, float shift,
                                          float* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int half = dim / 2;
  if (i >= m * half) return;
  const int row = i / half, j = i % half;
  const float expo = -logf(10000.0f) * static_cast<float>(j) / (static_cast<float>(half) - shift);
  const float arg = t[row] * expf(expo);
  const float s = sinf(arg), c = cosf(arg);
  float* o = out + static_cast<long long>(row) * dim;
  if (flip) o[j] = c, o[half + j] = s;
  else o[j] = s, o[half + j] = c;
  if ((dim & 1) && j == 0) o[dim - 1] = 0.f;
}

// Embedder (embedder.py:15-40): out = [x, sin(x*1), cos(x*1), sin(x*2), cos(x*2), ...], freq = 2^k
__global__ void fourier_kernel(const float* __restrict__ x, long long rows, int d, int nf, float* __restrict__ out) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= rows * d) return;
  const long long row = i / d;
  const int j = static_cast<int>(i % d);
  const float v = x[i];
  float* o = out + row * (d * (1 + 2 * nf));
  o[j] = v;
  float freq = 1.0f;
  for (int k = 0; k < nf; ++k) {
    o[d * (1 + 2 * k) + j] = sinf(v * freq);
    o[d * (2 + 2 * k) + j] = cosf(v * freq);
    freq *= 2.0f;
  }
}

__device__ __forceinline__ float silu_f(float x) { return x / (1.0f + expf(-x)); }

// Skinny linear: CTA = 8 warps x 4 columns; activations staged once per CTA in shared memory (fp32), weights bf16
// streamed with 16-byte loads; rows processed in chunks of 16.
constexpr int LS_ROWS = 16;
__global__ void linear_small_kernel(const float* __restrict__ in, int m, int k, int ldi, const __nv_bfloat16* __restrict__ w,
                                    int ldw, const float* __restrict__ bias, int n, int pre_silu, int post_silu,
                                    float* __restrict__ out, int ldo) {
  extern __shared__ float s_in[];  // [LS_ROWS][k]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int col_base = blockIdx.x * 32 + warp * 4;
  for (int m0 = blockIdx.y * LS_ROWS; m0 < m; m0 += gridDim.y * LS_ROWS) {
    const int mrows = min(LS_ROWS, m - m0);
    __syncthreads();
    for (int i = threadIdx.x; i < mrows * k; i += blockDim.x) {
      const int r = i / k, c = i % k;
      float v = in[static_cast<long long>(m0 + r) * ldi + c];
      s_in[r * k + c] = pre_silu ? silu_f(v) : v;
    }
    __syncthreads();
    for (int cc = 0; cc < 4; ++cc) {
      const int col = col_base + cc;
      if (col >= n) break;
      float acc[LS_ROWS];
#pragma unroll
      for (int r = 0; r < LS_ROWS; ++r) acc[r] = 0.f;
      const __nv_bfloat16* wr = w + static_cast<long long>(col) * ldw;
      for (int kk = lane * 8; kk < k; kk += 256) {
        float wf[8];
        if (kk + 8 <= k && (ldw % 8) == 0) {
          const uint4 u = __ldg(reinterpret_cast<const uint4*>(wr + kk));
          const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&u);
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const float2 t = __bfloat1622float2(h[j]);
            wf[2 * j] = t.x, wf[2 * j + 1] = t.y;
          }
        } else {
#pragma unroll
          for (int j = 0; j < 8; ++j) wf[j] = (kk + j < k) ? __bfloat162float(wr[kk + j]) : 0.f;
        }
#pragma unroll
        for (int r = 0; r < LS_ROWS; ++r) {
          if (r < mrows) {
            const float* si = s_in + r * k + kk;
#pragma unroll
            for (int j = 0; j < 8; ++j)
              if (kk + j < k) acc[r] += wf[j] * si[j];
          }
        }
      }
#pragma unroll
      for (int r = 0; r < LS_ROWS; ++r) {
        float v = acc[r];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if (lane == 0 && r < mrows) {
          v += bias ? bias[col] : 0.f;
          out[static_cast<long long>(m0 + r) * ldo + col] = post_silu ? silu_f(v) : v;
        }
      }
    }
  }
}

// Direct convolution, one thread per output element (output channel fastest), fp32 accumulate.  Weights are [kh][kw][cin][cout]:
// the threads of a warp (consecutive output channels of one pixel) read consecutive weights and broadcast-read the same input
// value.  (With [cout][kh][kw][cin] weights every lane walked its own row, 32 sectors per load: the BEV-map encoder took
// 12.9 ms of the 15.3 ms a re-conditioning call costs, profiles/time_prepare_r2.txt.)
template <typename TI>
__global__ void conv_direct_kernel(const TI* __restrict__ x, int n, int h, int w, int cin, const float* __restrict__ wgt,
                                   const float* __restrict__ bias, int cout, int kh, int kw, int sh, int sw, int ph,
                                   int pw, int ho, int wo, int silu, const void* __restrict__ residual, void* __restrict__ out,
                                   int out_is_f32) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  const long long total = static_cast<long long>(n) * ho * wo * cout;
  if (i >= total) return;
  const int co = static_cast<int>(i % cout);
  long long p = i / cout;
  const int ow = static_cast<int>(p % wo);
  p /= wo;
  const int oh = static_cast<int>(p % ho);
  const int img = static_cast<int>(p / ho);
  float acc = bias ? bias[co] : 0.f;
  for (int r = 0; r < kh; ++r) {
    const int ih = oh * sh + r - ph;
    if (ih < 0 || ih >= h) continue;
    for (int s = 0; s < kw; ++s) {
      const int iw = ow * sw + s - pw;
      if (iw < 0 || iw >= w) continue;
      const TI* xp = x + ((static_cast<long long>(img) * h + ih) * w + iw) * cin;
      const float* wp = wgt + static_cast<long long>(r * kw + s) * cin * cout + co;
#pragma unroll 4
      for (int c = 0; c < cin; ++c) acc += ldf(xp + c) * __ldg(wp + static_cast<long long>(c) * cout);
    }
  }
  if (silu) acc = silu_f(acc);
  if (out_is_f32) {
    if (residual) acc += static_cast<const float*>(residual)[i];
    static_cast<float*>(out)[i] = acc;
  } else {
    if (residual) acc += __bfloat162float(static_cast<const __nv_bfloat16*>(residual)[i]);
    static_cast<__nv_bfloat16*>(out)[i] = __float2bfloat16_rn(acc);
  }
}

__global__ void cfg_ddim_kernel(const float* __restrict__ eps, int cfg, float guidance, const float* __restrict__ coef,
                                float* __restrict__ lat, long long n, int c, int eps_ld) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const long long pix = i / c;
  const int ch = static_cast<int>(i - pix * c);
  const long long npix = n / c;
  float e = eps[pix * eps_ld + ch];
  if (cfg) {
    const float ec = eps[(npix + pix) * eps_ld + ch];
    e = e + guidance * (ec - e);
  }
  lat[i] = coef[0] * lat[i] + coef[1] * e;
}

// Guidance combine + one UniPC (order <= 2, bh2, x0-prediction) step: every update of the multistep scheduler is a
// linear combination of  x, the previous corrected sample, and the last two x0 predictions  with per-step scalar
// coefficients (host: pipeline.UniPCSchedule), so corrector + history shift + predictor are one pass over the latents.
__global__ void cfg_unipc_kernel(const float* __restrict__ eps, int cfg, float guidance, const float* __restrict__ coef,
                                 float* __restrict__ lat, float* __restrict__ last, float* __restrict__ m0,
                                 float* __restrict__ m1, long long n, int c, int eps_ld) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const long long pix = i / c;
  const int ch = static_cast<int>(i - pix * c);
  const long long npix = n / c;
  float e = eps[pix * eps_ld + ch];
  if (cfg) {
    const float ec = eps[(npix + pix) * eps_ld + ch];
    e = e + guidance * (ec - e);
  }
  const float x = lat[i], h0 = m0[i], h1 = m1[i];
  const float x0 = coef[0] * x + coef[1] * e;                                                   // convert_model_output
  const float xc = (coef[9] != 0.f) ? coef[2] * last[i] + coef[3] * h0 + coef[4] * h1 + coef[5] * x0 : x;  // UniC
  lat[i] = coef[6] * xc + coef[7] * x0 + coef[8] * h0;                                          // UniP
  last[i] = xc;
  m1[i] = h0;
  m0[i] = x0;
}

// rows of the views flagged in view_mask: dst = coef[0] * a + coef[1] * b  (a may be null).  Serves the given-view
// pipeline: re-noising pinned views (a = clean latents, b = their initial noise, coef = sqrt(abar_t), sqrt(1 - abar_t))
// and replacing their predicted noise by the initial noise (a = null, coef = {0, 1}).
__global__ void pin_views_kernel(float* __restrict__ dst, int dst_ld, const float* __restrict__ a,
                                 const float* __restrict__ b, int c, const float* __restrict__ coef,
                                 const int* __restrict__ view_mask, long long rows_per_view, long long n) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const long long row = i / c;
  const int ch = static_cast<int>(i - row * c);
  if (!view_mask[row / rows_per_view]) return;
  float v = coef[1] * b[i];
  if (a) v += coef[0] * a[i];
  dst[row * dst_ld + ch] = v;
}

// latents [pix, cin] (fp32 or bf16) -> bf16 [repeat * pix, cpad], channels >= cin zero: the K-padded A operand of the
// tensor-core conv_in; `repeat` = 2 duplicates the batch for classifier-free guidance ([uncond ; cond] share latents)
template <typename TI>
__global__ void pack_latents_kernel(const TI* __restrict__ x, long long pix, int cin, int cpad, int repeat,
                                    __nv_bfloat16* __restrict__ out) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= pix * cpad) return;
  const long long p = i / cpad;
  const int c = static_cast<int>(i - p * cpad);
  const __nv_bfloat16 v = (c < cin) ? __float2bfloat16_rn(ldf(x + p * cin + c)) : __float2bfloat16_rn(0.f);
  for (int r = 0; r < repeat; ++r) out[(r * pix + p) * cpad + c] = v;
}

// NCHW images [n, cin, h, w] (fp32 or bf16) -> bf16 [n*h*w, 64]: row = output pixel, column (r*3 + s)*cin + c = input
// channel c at tap (r, s) of the zero-padded 3x3 neighbourhood, columns >= 9*cin zero.  The encoder's conv_in then runs
// as one K = 64 GEMM.  A block stages a (TH + 2) x (TW + 2) halo tile of every channel in shared memory (each input
// element is read from global memory once per tile) and writes each of its pixels as one 128-byte row: 8 threads x 16 bytes.
constexpr int PATCH_TW = 32, PATCH_TH = 8, PATCH_MAXC = 7;
template <typename TI>
__global__ void __launch_bounds__(256) pack_image_patches_kernel(const TI* __restrict__ x, int cin, int h, int w,
                                                                 uint4* __restrict__ out) {
  __shared__ float tile[PATCH_MAXC][PATCH_TH + 2][PATCH_TW + 2];
  const int img = blockIdx.z, y0 = blockIdx.y * PATCH_TH, x0 = blockIdx.x * PATCH_TW;
  const TI* xi = x + static_cast<long long>(img) * cin * h * w;
  constexpr int per_c = (PATCH_TH + 2) * (PATCH_TW + 2);
  for (int i = threadIdx.x; i < cin * per_c; i += blockDim.x) {
    const int c = i / per_c, rem = i - c * per_c;
    const int r = rem / (PATCH_TW + 2), s = rem - r * (PATCH_TW + 2);
    const int yy = y0 + r - 1, xx = x0 + s - 1;
    tile[c][r][s] = (yy >= 0 && yy < h && xx >= 0 && xx < w) ? ldf(xi + (static_cast<long long>(c) * h + yy) * w + xx) : 0.f;
  }
  __syncthreads();
  const int px = threadIdx.x >> 3, q = threadIdx.x & 7;  // pixel of the tile row, 16-byte chunk of its output row
  const int xx = x0 + px;
  if (xx >= w) return;
  const int kcols = 9 * cin;
  for (int r = 0; r < PATCH_TH && y0 + r < h; ++r) {
    __align__(16) __nv_bfloat16 v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int col = q * 8 + j;
      float f = 0.f;
      if (col < kcols) {
        const int tap = col / cin, c = col - tap * cin;
        f = tile[c][r + tap / 3][px + tap % 3];
      }
      v[j] = __float2bfloat16_rn(f);
    }
    out[((static_cast<long long>(img) * h + y0 + r) * w + xx) * 8 + q] = *reinterpret_cast<const uint4*>(v);
  }
}

// DiagonalGaussianDistribution of the encoder's moments: NHWC fp32 [pix, ldm] rows (mean[0:c] | logvar[c:2c]) -> NCHW fp32
// [n, c, h, w] = scale * (mean + exp(0.5 * clamp(logvar, -30, 20)) * noise), noise NCHW like the output (null: scale * mean).
__global__ void latent_dist_kernel(const float* __restrict__ mom, int ldm, int c, long long hw, long long total,
                                   const float* __restrict__ noise, float scale, float* __restrict__ out) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const long long nc = i / hw, p = i - nc * hw;
  const long long img = nc / c;
  const int ch = static_cast<int>(nc - img * c);
  const float* m = mom + (img * hw + p) * ldm;
  float v = m[ch];
  if (noise) {
    const float lv = fminf(fmaxf(m[c + ch], -30.f), 20.f);
    v += expf(0.5f * lv) * noise[i];
  }
  out[i] = scale * v;
}

inline unsigned nblocks(long long n, int t) { return static_cast<unsigned>((n + t - 1) / t); }

}  // namespace

using namespace mdb;

extern "C" int mdb_add(const void* a, const void* b, void* out, long long n, void* stream) {
  if (!a || !b || !out) return set_error(MDB_ERR_INVALID, "mdb_add: null pointer");
  if (n % 8) return set_error(MDB_ERR_UNSUPPORTED, "mdb_add: n must be a multiple of 8");
  add_kernel<<<nblocks(n / 8, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const uint4*>(a), static_cast<const uint4*>(b), static_cast<uint4*>(out), n / 8);
  MDB_CHECK_LAUNCH("add_kernel");
  return MDB_OK;
}

extern "C" int mdb_upsample_nearest(const void* x, int n, int h, int w, int c, void* out, int ho, int wo, void* stream) {
  if (!x || !out) return set_error(MDB_ERR_INVALID, "mdb_upsample_nearest: null pointer");
  if (c % 8) return set_error(MDB_ERR_UNSUPPORTED, "mdb_upsample_nearest: c must be a multiple of 8");
  const long long total = static_cast<long long>(n) * ho * wo * (c / 8);
  upsample_nearest_kernel<<<nblocks(total, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const uint4*>(x), n, h, w, c / 8, static_cast<uint4*>(out), ho, wo);
  MDB_CHECK_LAUNCH("upsample_nearest_kernel");
  return MDB_OK;
}

extern "C" int mdb_adaptive_avgpool(const float* x, int n, int h, int w, int c, float* out, int ho, int wo, int silu, void* stream) {
  if (!x || !out) return set_error(MDB_ERR_INVALID, "mdb_adaptive_avgpool: null pointer");
  if (n <= 0 || h <= 0 || w <= 0 || c <= 0 || ho <= 0 || wo <= 0) return set_error(MDB_ERR_INVALID, "mdb_adaptive_avgpool: bad shape");
  const long long total = static_cast<long long>(n) * ho * wo * c;
  adaptive_avgpool_kernel<<<nblocks(total, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(x, n, h, w, c, out, ho, wo, silu);
  MDB_CHECK_LAUNCH("adaptive_avgpool_kernel");
  return MDB_OK;
}

extern "C" int mdb_nchw_to_nhwc(const void* x, int x_is_f32, int n, int c, int h, int w, void* out, void* stream) {
  if (!x || !out) return set_error(MDB_ERR_INVALID, "mdb_nchw_to_nhwc: null pointer");
  const int hw = h * w;
  dim3 grid((hw + 31) / 32, (c + 31) / 32, n), block(32, 8);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (x_is_f32)
    nchw_to_nhwc_kernel<float><<<grid, block, 0, st>>>(static_cast<const float*>(x), c, hw, static_cast<__nv_bfloat16*>(out));
  else
    nchw_to_nhwc_kernel<__nv_bfloat16><<<grid, block, 0, st>>>(static_cast<const __nv_bfloat16*>(x), c, hw,
                                                               static_cast<__nv_bfloat16*>(out));
  MDB_CHECK_LAUNCH("nchw_to_nhwc_kernel");
  return MDB_OK;
}

extern "C" int mdb_nhwc_to_nchw(const void* x, int n, int c, int h, int w, void* out, int out_is_f32, void* stream) {
  if (!x || !out) return set_error(MDB_ERR_INVALID, "mdb_nhwc_to_nchw: null pointer");
  const int hw = h * w;
  dim3 grid((hw + 31) / 32, (c + 31) / 32, n), block(32, 8);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (out_is_f32)
    nhwc_to_nchw_kernel<float><<<grid, block, 0, st>>>(static_cast<const __nv_bfloat16*>(x), c, hw, static_cast<float*>(out));
  else
    nhwc_to_nchw_kernel<__nv_bfloat16><<<grid, block, 0, st>>>(static_cast<const __nv_bfloat16*>(x), c, hw,
                                                               static_cast<__nv_bfloat16*>(out));
  MDB_CHECK_LAUNCH("nhwc_to_nchw_kernel");
  return MDB_OK;
}

extern "C" int mdb_f32_to_bf16(const float* x, void* out, long long n, void* stream) {
  if (!x || !out) return set_error(MDB_ERR_INVALID, "mdb_f32_to_bf16: null pointer");
  f32_to_bf16_kernel<<<nblocks(n, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(x, static_cast<__nv_bfloat16*>(out), n);
  MDB_CHECK_LAUNCH("f32_to_bf16_kernel");
  return MDB_OK;
}
extern "C" int mdb_bf16_to_f32(const void* x, float* out, long long n, void* stream) {
  if (!x || !out) return set_error(MDB_ERR_INVALID, "mdb_bf16_to_f32: null pointer");
  bf16_to_f32_kernel<<<nblocks(n, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(static_cast<const __nv_bfloat16*>(x), out, n);
  MDB_CHECK_LAUNCH("bf16_to_f32_kernel");
  return MDB_OK;
}

extern "C" int mdb_timestep_embedding(const float* t, int m, int dim, int flip_sin_to_cos, float freq_shift, float* out,
                                      void* stream) {
  if (!t || !out) return set_error(MDB_ERR_INVALID, "mdb_timestep_embedding: null pointer");
  timestep_embedding_kernel<<<nblocks(static_cast<long long>(m) * (dim / 2), 128), 128, 0, static_cast<cudaStream_t>(stream)>>>(
      t, m, dim, flip_sin_to_cos, freq_shift, out);
  MDB_CHECK_LAUNCH("timestep_embedding_kernel");
  return MDB_OK;
}

extern "C" int mdb_fourier_embed(const float* x, long long rows, int d, int num_freqs, float* out, void* stream) {
  if (!x || !out) return set_error(MDB_ERR_INVALID, "mdb_fourier_embed: null pointer");
  fourier_kernel<<<nblocks(rows * d, 128), 128, 0, static_cast<cudaStream_t>(stream)>>>(x, rows, d, num_freqs, out);
  MDB_CHECK_LAUNCH("fourier_kernel");
  return MDB_OK;
}

extern "C" int mdb_linear_small(const float* in, int m, int k, int ldi, const void* w, int ldw, const float* bias, int n,
                                int pre_silu, int post_silu, float* out, int ldo, void* stream) {
  if (!in || !w || !out) return set_error(MDB_ERR_INVALID, "mdb_linear_small: null pointer");
  const size_t smem = sizeof(float) * LS_ROWS * k;
  if (smem > 200 * 1024) return set_error(MDB_ERR_UNSUPPORTED, "mdb_linear_small: k=%d too large", k);
  static bool attr = false;
  if (!attr) {
    cudaFuncSetAttribute(linear_small_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    attr = true;
  }
  int gy = (m + LS_ROWS - 1) / LS_ROWS;
  if (gy > 64) gy = 64;
  dim3 grid((n + 31) / 32, gy);
  linear_small_kernel<<<grid, 256, smem, static_cast<cudaStream_t>(stream)>>>(
      in, m, k, ldi, static_cast<const __nv_bfloat16*>(w), ldw, bias, n, pre_silu, post_silu, out, ldo);
  MDB_CHECK_LAUNCH("linear_small_kernel");
  return MDB_OK;
}

extern "C" int mdb_conv_direct(const void* x, int x_is_f32, int n, int h, int w, int cin, const float* wgt, const float* bias,
                               int cout, int kh, int kw, int stride_h, int stride_w, int pad_h, int pad_w, int ho, int wo,
                               int silu, const void* residual, void* out, int out_is_f32, void* stream) {
  if (!x || !wgt || !out) return set_error(MDB_ERR_INVALID, "mdb_conv_direct: null pointer");
  const long long total = static_cast<long long>(n) * ho * wo * cout;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (x_is_f32)
    conv_direct_kernel<float><<<nblocks(total, 128), 128, 0, st>>>(static_cast<const float*>(x), n, h, w, cin, wgt, bias, cout,
                                                                   kh, kw, stride_h, stride_w, pad_h, pad_w, ho, wo, silu,
                                                                   residual, out, out_is_f32);
  else
    conv_direct_kernel<__nv_bfloat16><<<nblocks(total, 128), 128, 0, st>>>(
        static_cast<const __nv_bfloat16*>(x), n, h, w, cin, wgt, bias, cout, kh, kw, stride_h, stride_w, pad_h, pad_w, ho, wo,
        silu, residual, out, out_is_f32);
  MDB_CHECK_LAUNCH("conv_direct_kernel");
  return MDB_OK;
}

extern "C" int mdb_pack_latents(const void* x, int x_is_f32, long long pix, int cin, int cpad, int repeat, void* out,
                                void* stream) {
  if (!x || !out) return set_error(MDB_ERR_INVALID, "mdb_pack_latents: null pointer");
  if (cpad < cin || repeat < 1) return set_error(MDB_ERR_INVALID, "mdb_pack_latents: bad shape");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (x_is_f32)
    pack_latents_kernel<float><<<nblocks(pix * cpad, 256), 256, 0, st>>>(static_cast<const float*>(x), pix, cin, cpad, repeat,
                                                                         static_cast<__nv_bfloat16*>(out));
  else
    pack_latents_kernel<__nv_bfloat16><<<nblocks(pix * cpad, 256), 256, 0, st>>>(
        static_cast<const __nv_bfloat16*>(x), pix, cin, cpad, repeat, static_cast<__nv_bfloat16*>(out));
  MDB_CHECK_LAUNCH("pack_latents_kernel");
  return MDB_OK;
}

extern "C" int mdb_pack_image_patches(const void* x, int x_is_f32, int n, int cin, int h, int w, void* out, void* stream) {
  if (!x || !out) return set_error(MDB_ERR_INVALID, "mdb_pack_image_patches: null pointer");
  if (n <= 0 || h <= 0 || w <= 0 || cin < 1 || cin > PATCH_MAXC)
    return set_error(MDB_ERR_INVALID, "mdb_pack_image_patches: bad shape (n=%d cin=%d h=%d w=%d; 9*cin must fit 64 columns)",
                     n, cin, h, w);
  if (reinterpret_cast<uintptr_t>(out) & 15) return set_error(MDB_ERR_INVALID, "mdb_pack_image_patches: out must be 16-byte aligned");
  dim3 grid((w + PATCH_TW - 1) / PATCH_TW, (h + PATCH_TH - 1) / PATCH_TH, n);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (x_is_f32)
    pack_image_patches_kernel<float><<<grid, 256, 0, st>>>(static_cast<const float*>(x), cin, h, w, static_cast<uint4*>(out));
  else
    pack_image_patches_kernel<__nv_bfloat16><<<grid, 256, 0, st>>>(static_cast<const __nv_bfloat16*>(x), cin, h, w,
                                                                    static_cast<uint4*>(out));
  MDB_CHECK_LAUNCH("pack_image_patches_kernel");
  return MDB_OK;
}

extern "C" int mdb_latent_dist(const float* moments, int ldm, int n, int c, int h, int w, const float* noise, float scale,
                               float* out, void* stream) {
  if (!moments || !out) return set_error(MDB_ERR_INVALID, "mdb_latent_dist: null pointer");
  if (n <= 0 || c <= 0 || h <= 0 || w <= 0 || ldm < 2 * c) return set_error(MDB_ERR_INVALID, "mdb_latent_dist: bad shape");
  const long long hw = static_cast<long long>(h) * w, total = static_cast<long long>(n) * c * hw;
  latent_dist_kernel<<<nblocks(total, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(moments, ldm, c, hw, total, noise,
                                                                                         scale, out);
  MDB_CHECK_LAUNCH("latent_dist_kernel");
  return MDB_OK;
}

extern "C" int mdb_cfg_ddim_step(const float* eps, int eps_ld, int c, int cfg, float guidance, const float* coef,
                                 float* latents, long long n, void* stream) {
  if (!eps || !coef || !latents) return set_error(MDB_ERR_INVALID, "mdb_cfg_ddim_step: null pointer");
  if (c <= 0 || eps_ld < c || n % c) return set_error(MDB_ERR_INVALID, "mdb_cfg_ddim_step: bad shape");
  cfg_ddim_kernel<<<nblocks(n, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(eps, cfg, guidance, coef, latents, n, c,
                                                                                  eps_ld);
  MDB_CHECK_LAUNCH("cfg_ddim_kernel");
  return MDB_OK;
}

extern "C" int mdb_cfg_unipc_step(const float* eps, int eps_ld, int c, int cfg, float guidance, const float* coef,
                                  float* latents, float* last_sample, float* m0, float* m1, long long n, void* stream) {
  if (!eps || !coef || !latents || !last_sample || !m0 || !m1)
    return set_error(MDB_ERR_INVALID, "mdb_cfg_unipc_step: null pointer");
  if (c <= 0 || eps_ld < c || n % c) return set_error(MDB_ERR_INVALID, "mdb_cfg_unipc_step: bad shape");
  cfg_unipc_kernel<<<nblocks(n, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(eps, cfg, guidance, coef, latents,
                                                                                   last_sample, m0, m1, n, c, eps_ld);
  MDB_CHECK_LAUNCH("cfg_unipc_kernel");
  return MDB_OK;
}

extern "C" int mdb_pin_views(float* dst, int dst_ld, const float* a, const float* b, int c, const float* coef,
                             const int* view_mask, long long rows_per_view, int n_views, void* stream) {
  if (!dst || !b || !coef || !view_mask) return set_error(MDB_ERR_INVALID, "mdb_pin_views: null pointer");
  if (c <= 0 || dst_ld < c || rows_per_view <= 0 || n_views <= 0) return set_error(MDB_ERR_INVALID, "mdb_pin_views: bad shape");
  const long long n = rows_per_view * n_views * c;
  pin_views_kernel<<<nblocks(n, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(dst, dst_ld, a, b, c, coef, view_mask,
                                                                                   rows_per_view, n);
  MDB_CHECK_LAUNCH("pin_views_kernel");
  return MDB_OK;
}
