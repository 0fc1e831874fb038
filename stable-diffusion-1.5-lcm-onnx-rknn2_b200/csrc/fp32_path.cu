// fp32 precision mode (reference `CUDA_DTYPE=fp32`, `backends/cuda_worker.py:55-61`): the same hot
// path with fp32 activations and weights on the CUDA cores.  It exists for the parity bar of the
// spec (per-step noise_pred within 1e-4 of the fp32 pipeline), not for speed: plain tiled SIMT
// kernels, accurate expf / erff / tanh-free SiLU, fp32 accumulation everywhere.  The bf16
// tcgen05 path is the product path; these entry points mirror its C-ABI one to one so the host
// engine is shared (the binding dispatches on the tensor dtype).
#include <math.h>
#include <string.h>

#include "common.cuh"
#include "dreamlab_b200.h"

namespace dl {

// ------------------------------------------------------------------------------------------------
// implicit-GEMM conv / linear:  out[pixel, n] = epi( sum_{tap, c} a[pixel + off(tap), c] * w[n, tap, c] )
// 64 pixels x 64 output channels per CTA, K chunks of 16, 256 threads with 4 x 4 outputs each.
// ------------------------------------------------------------------------------------------------
struct F32GemmParams {
  const float* a0; long long a0_ps; int c0;
  const float* a1; long long a1_ps; int c1;
  int nimg, h, w, taps, in_rows, in_row0;
  signed char tdy[9], tdx[9];
  const float* wgt; long long ldw; int n;
  void* out; long long ldo, osx, osy, osi;
  const float* bias; const float* rowadd; int ld_rowadd;
  const float* residual; long long ldr;
  int mode; float alpha;
};

constexpr int FT = 64, FK = 16;

__device__ __forceinline__ float gelu_exact(float x) { return 0.5f * x * (1.0f + erff(x * 0.70710678118654752f)); }
__device__ __forceinline__ float silu_exact(float x) { return x / (1.0f + expf(-x)); }

__global__ void __launch_bounds__(256) f32_gemm_kernel(const F32GemmParams p) {
  __shared__ float As[FK][FT + 4];
  __shared__ float Bs[FK][FT + 4];
  const int t = threadIdx.x;
  const long long M = (long long)p.nimg * p.h * p.w;
  const long long m0 = (long long)blockIdx.x * FT;
  const int n0 = blockIdx.y * FT;
  const int C = p.c0 + p.c1;
  const int K = p.taps * C;
  // loader roles: one float4 of A (pixel lp, channels lq*4..) and one of B (column lp, k lq*4..)
  const int lp = t >> 2, lq = t & 3;
  const long long lm = m0 + lp;
  int l_img = 0, l_y = 0, l_x = 0;
  const bool lm_ok = lm < M;
  if (lm_ok) {
    l_img = (int)(lm / ((long long)p.h * p.w));
    const int rem = (int)(lm - (long long)l_img * p.h * p.w);
    l_y = rem / p.w;
    l_x = rem - l_y * p.w;
  }
  const int ty = t >> 4, tx = t & 15;
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

  for (int k0 = 0; k0 < K; k0 += FK) {
    const int tap = k0 / C;
    const int cc = k0 - tap * C + lq * 4;                 // channel of the virtual concat
    float4 av = make_float4(0.f, 0.f, 0.f, 0.f);
    if (lm_ok) {
      const int yi = l_y + p.tdy[tap] + p.in_row0, xi = l_x + p.tdx[tap];
      if (yi >= 0 && yi < p.in_rows && xi >= 0 && xi < p.w) {
        const long long pix = ((long long)l_img * p.in_rows + yi) * p.w + xi;
        av = (cc < p.c0) ? *reinterpret_cast<const float4*>(p.a0 + pix * p.a0_ps + cc)
                         : *reinterpret_cast<const float4*>(p.a1 + pix * p.a1_ps + (cc - p.c0));
      }
    }
    float4 bv = make_float4(0.f, 0.f, 0.f, 0.f);
    if (n0 + lp < p.n) bv = *reinterpret_cast<const float4*>(p.wgt + (long long)(n0 + lp) * p.ldw + k0 + lq * 4);
    __syncthreads();
    As[lq * 4 + 0][lp] = av.x; As[lq * 4 + 1][lp] = av.y; As[lq * 4 + 2][lp] = av.z; As[lq * 4 + 3][lp] = av.w;
    Bs[lq * 4 + 0][lp] = bv.x; Bs[lq * 4 + 1][lp] = bv.y; Bs[lq * 4 + 2][lp] = bv.z; Bs[lq * 4 + 3][lp] = bv.w;
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < FK; ++kk) {
      const float4 a = *reinterpret_cast<const float4*>(&As[kk][ty * 4]);
      const float4 b = *reinterpret_cast<const float4*>(&Bs[kk][tx * 4]);
      const float ar[4] = {a.x, a.y, a.z, a.w}, br[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(ar[i], br[j], acc[i][j]);
    }
  }
  // ---- epilogue ----
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const long long m = m0 + ty * 4 + i;
    if (m >= M) continue;
    const int img = (int)(m / ((long long)p.h * p.w));
    const int rem = (int)(m - (long long)img * p.h * p.w);
    const int y = rem / p.w, x = rem - y * p.w;
    float v[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int col = n0 + tx * 4 + j;
      float r = acc[i][j] * p.alpha;
      if (col < p.n) {
        if (p.bias) r += p.bias[col];
        if (p.rowadd) r += p.rowadd[(long long)img * p.ld_rowadd + col];
        if (p.residual) r += p.residual[m * p.ldr + col];
      }
      v[j] = r;
    }
    const long long obase = (long long)img * p.osi + (long long)y * p.osy + (long long)x * p.osx;
    if (p.mode == DL_EPI_GEGLU) {
      // interleaved columns (value, gate): 2 outputs from this thread's 4 accumulators
#pragma unroll
      for (int j = 0; j < 4; j += 2) {
        const int col = n0 + tx * 4 + j;
        if (col + 1 < p.n)
          reinterpret_cast<float*>(p.out)[obase + (col >> 1)] = v[j] * gelu_exact(v[j + 1]);
      }
    } else if (p.mode == DL_EPI_U8_IMAGE) {
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int col = n0 + tx * 4 + j;
        if (col < p.n) {
          const float f = fminf(fmaxf(v[j] * 0.5f + 0.5f, 0.0f), 1.0f) * 255.0f;
          reinterpret_cast<uint8_t*>(p.out)[obase + col] = (uint8_t)__float2int_rn(f);
        }
      }
    } else {
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int col = n0 + tx * 4 + j;
        if (col < p.n) reinterpret_cast<float*>(p.out)[obase + col] = v[j];
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// GroupNorm(+SiLU) fp32, optional two-source concat: one CTA per (image, group), two-pass stats
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) f32_groupnorm_kernel(const float* __restrict__ x0, int c0,
                                                            const float* __restrict__ x1, int c1, int hw,
                                                            int groups, float eps, const float* __restrict__ gamma,
                                                            const float* __restrict__ beta, int apply_silu,
                                                            float* __restrict__ out) {
  __shared__ float red[256];
  __shared__ float s_stat[2];
  const int C = c0 + c1, cpg = C / groups;
  const int img = blockIdx.y, g = blockIdx.x;
  const long long n = (long long)hw * cpg;
  auto load = [&](long long i) -> float {
    const int px = (int)(i / cpg), c = g * cpg + (int)(i - (long long)px * cpg);
    const long long pix = (long long)img * hw + px;
    return c < c0 ? x0[pix * c0 + c] : x1[pix * c1 + (c - c0)];
  };
  auto block_sum = [&](float v) -> float {
    red[threadIdx.x] = v;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
      if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
      __syncthreads();
    }
    const float r = red[0];
    __syncthreads();
    return r;
  };
  float s = 0.f;
  for (long long i = threadIdx.x; i < n; i += 256) s += load(i);
  const float mean = block_sum(s) / (float)n;
  float q = 0.f;
  for (long long i = threadIdx.x; i < n; i += 256) { const float d = load(i) - mean; q = fmaf(d, d, q); }
  const float rstd = rsqrtf(block_sum(q) / (float)n + eps);
  (void)s_stat;
  for (long long i = threadIdx.x; i < n; i += 256) {
    const int px = (int)(i / cpg), c = g * cpg + (int)(i - (long long)px * cpg);
    float v = (load(i) - mean) * rstd * gamma[c] + beta[c];
    if (apply_silu) v = silu_exact(v);
    out[((long long)img * hw + px) * C + c] = v;
  }
}

// LayerNorm fp32: one warp per row, two-pass
__global__ void f32_layernorm_kernel(const float* __restrict__ x, long long rows, int C, float eps,
                                     const float* __restrict__ gamma, const float* __restrict__ beta,
                                     float* __restrict__ out) {
  const long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int lane = threadIdx.x & 31;
  const float* xr = x + row * C;
  float s = 0.f;
  for (int c = lane; c < C; c += 32) s += xr[c];
  const float mean = warp_sum(s) / (float)C;
  float q = 0.f;
  for (int c = lane; c < C; c += 32) { const float d = xr[c] - mean; q = fmaf(d, d, q); }
  const float rstd = rsqrtf(warp_sum(q) / (float)C + eps);
  for (int c = lane; c < C; c += 32) out[row * C + c] = (xr[c] - mean) * rstd * gamma[c] + beta[c];
}

// attention fp32: one warp per query row, 32 keys per step, online softmax (expf), d <= 512
constexpr int FA_WARPS = 8, FA_KEYS = 32, FA_MAXD = 512;
__global__ void __launch_bounds__(FA_WARPS * 32)
f32_attention_kernel(const float* __restrict__ q, long long ldq, const float* __restrict__ k, long long ldk,
                     const float* __restrict__ v, long long ldv, int dh_stride, float* __restrict__ out,
                     long long ldo, int sq, int skv, int d, float scale, int causal) {
  extern __shared__ float sm[];
  const int dp = d + 1;
  float* sK = sm;
  float* sV = sK + FA_KEYS * dp;
  float* sQ = sV + FA_KEYS * dp;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int h = blockIdx.y, b = blockIdx.z;
  const int qi = blockIdx.x * FA_WARPS + warp;
  const bool active = qi < sq;
  const float* qrow = q + ((long long)b * sq + (active ? qi : 0)) * ldq + h * dh_stride;
  for (int i = lane; i < d; i += 32) sQ[warp * d + i] = qrow[i] * scale;
  constexpr int NACC = FA_MAXD / 32;
  float acc[NACC];
#pragma unroll
  for (int i = 0; i < NACC; ++i) acc[i] = 0.f;
  float m = -INFINITY, l = 0.f;
  for (int k0 = 0; k0 < skv; k0 += FA_KEYS) {
    __syncthreads();
    for (int idx = threadIdx.x; idx < FA_KEYS * d; idx += blockDim.x) {
      const int j = idx / d, i = idx % d;
      const bool ok = (k0 + j) < skv;
      const long long r = (long long)b * skv + k0 + j;
      sK[j * dp + i] = ok ? k[r * ldk + h * dh_stride + i] : 0.f;
      sV[j * dp + i] = ok ? v[r * ldv + h * dh_stride + i] : 0.f;
    }
    __syncthreads();
    float s = 0.f;
    for (int i = 0; i < d; ++i) s = fmaf(sQ[warp * d + i], sK[lane * dp + i], s);
    if (k0 + lane >= skv || (causal && k0 + lane > qi)) s = -INFINITY;
    const float m_new = fmaxf(m, warp_max(s));
    const float p = expf(s - m_new);
    const float corr = expf(m - m_new);
    l = l * corr + warp_sum(p);
    m = m_new;
#pragma unroll
    for (int i = 0; i < NACC; ++i) acc[i] *= corr;
    for (int j = 0; j < FA_KEYS; ++j) {
      const float pj = __shfl_sync(0xffffffffu, p, j);
#pragma unroll
      for (int i = 0; i < NACC; ++i) {
        const int dim = lane + 32 * i;
        if (dim < d) acc[i] = fmaf(pj, sV[j * dp + dim], acc[i]);
      }
    }
  }
  if (active) {
    float* orow = out + ((long long)b * sq + qi) * ldo + h * d;
    const float inv = 1.f / l;
#pragma unroll
    for (int i = 0; i < NACC; ++i) {
      const int dim = lane + 32 * i;
      if (dim < d) orow[dim] = acc[i] * inv;
    }
  }
}

// small pieces
__global__ void f32_pack_latent_kernel(const float* __restrict__ x, long long npix, int cin, int cpad, float scale,
                                       const float* __restrict__ mat, const float* __restrict__ vec,
                                       float* __restrict__ out) {
  const long long total = npix * cpad;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(i % cpad);
    const long long px = i / cpad;
    float r = 0.f;
    if (c < cin) {
      if (mat) {
        r = vec ? vec[c] : 0.f;
        for (int j = 0; j < cin; ++j) r += mat[c * cin + j] * (x[px * cin + j] * scale);
      } else {
        r = x[px * cin + c] * scale;
      }
    }
    out[i] = r;
  }
}

// pad = 1: symmetric padding 1; pad = 0: bottom / right zero pad (see im2col_s2_kernel)
__global__ void f32_im2col_s2_kernel(const float4* __restrict__ x, int nimg, int h, int w, int V,
                                     float4* __restrict__ cols, int pad) {
  const int ho = h / 2, wo = w / 2;
  const long long total = (long long)nimg * ho * wo * 9 * V;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int v = (int)(i % V);
    long long r = i / V;
    const int tap = (int)(r % 9);
    r /= 9;
    const int xo = (int)(r % wo);
    r /= wo;
    const int yo = (int)(r % ho);
    const int n = (int)(r / ho);
    const int yi = 2 * yo + tap / 3 - pad, xi = 2 * xo + tap % 3 - pad;
    float4 val = make_float4(0.f, 0.f, 0.f, 0.f);
    if (yi >= 0 && yi < h && xi >= 0 && xi < w) val = x[(((long long)n * h + yi) * w + xi) * V + v];
    cols[i] = val;
  }
}

__global__ void f32_softmax_rows_kernel(const float* __restrict__ s, long long rows, int cols,
                                        float* __restrict__ out) {
  __shared__ float red[256];
  const long long row = blockIdx.x;
  const float* r = s + row * cols;
  float mx = -INFINITY;
  for (int c = threadIdx.x; c < cols; c += 256) mx = fmaxf(mx, r[c]);
  red[threadIdx.x] = mx;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) { if (threadIdx.x < o) red[threadIdx.x] = fmaxf(red[threadIdx.x], red[threadIdx.x + o]); __syncthreads(); }
  mx = red[0];
  __syncthreads();
  float sum = 0.f;
  for (int c = threadIdx.x; c < cols; c += 256) sum += expf(r[c] - mx);
  red[threadIdx.x] = sum;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) { if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o]; __syncthreads(); }
  const float inv = 1.f / red[0];
  for (int c = threadIdx.x; c < cols; c += 256) out[row * cols + c] = expf(r[c] - mx) * inv;
}

// out[m,n] = act_out(sum_k act_in(x[m,k]) w[n,k] + bias[n] + add[m,n]), fp32 weights, exact SiLU
__global__ void f32_small_linear_kernel(const float* __restrict__ x, int m, int k, const float* __restrict__ w,
                                        const float* __restrict__ bias, const float* __restrict__ add, int n,
                                        int silu_in, int silu_out, float* __restrict__ out) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= n * m) return;
  const int col = warp % n, row = warp / n;
  float s = 0.f;
  for (int i = lane; i < k; i += 32) {
    float xv = x[(long long)row * k + i];
    if (silu_in) xv = silu_exact(xv);
    s = fmaf(xv, w[(long long)col * k + i], s);
  }
  s = warp_sum(s);
  if (lane == 0) {
    float r = s + (bias ? bias[col] : 0.f) + (add ? add[(long long)row * n + col] : 0.f);
    if (silu_out) r = silu_exact(r);
    out[(long long)row * n + col] = r;
  }
}

static inline unsigned f32_grid(long long total, int threads) {
  long long b = (total + threads - 1) / threads;
  const long long cap = (long long)num_sms() * 32;
  if (b > cap) b = cap;
  if (b < 1) b = 1;
  return (unsigned)b;
}

}  // namespace dl

using namespace dl;
#define STREAM reinterpret_cast<cudaStream_t>(stream_)

extern "C" int dl_igemm_f32(const dl_igemm_desc* d, void* stream_) {
  DL_CHECK_ARG(d->a0 && d->wgt && d->out, "igemm_f32: null pointer");
  DL_CHECK_ARG(d->taps == 1 || d->taps == 9 || (d->taps == 4 && d->tap_phase >= 0 && d->tap_phase < 4),
               "igemm_f32: taps must be 1, 9, or 4 with tap_phase");
  DL_CHECK_ARG(d->c0 > 0 && d->c0 % 16 == 0 && d->c1 % 16 == 0, "igemm_f32: channels must be multiples of 16");
  DL_CHECK_ARG(d->mode >= 0 && d->mode <= DL_EPI_U8_IMAGE, "igemm_f32: bad epilogue mode");
  // the fused statistics and peer stores of the bf16 kernel have no fp32 counterpart: refuse them
  // rather than leave the caller's buffers unwritten
  DL_CHECK_ARG(!d->gn_partial, "igemm_f32: the fp32 mode has no fused GroupNorm statistics (gn_partial)");
  DL_CHECK_ARG(!d->row_stats_out, "igemm_f32: the fp32 mode has no fused row statistics (row_stats_out)");
  DL_CHECK_ARG(!d->ln_stats, "igemm_f32: the fp32 mode has no folded LayerNorm statistics (ln_stats)");
  DL_CHECK_ARG(d->n_peer_out == 0, "igemm_f32: the fp32 mode has no peer stores (n_peer_out=%d)", d->n_peer_out);
  F32GemmParams p;
  memset(&p, 0, sizeof(p));
  p.a0 = reinterpret_cast<const float*>(d->a0); p.a0_ps = d->a0_pix_stride; p.c0 = d->c0;
  p.a1 = reinterpret_cast<const float*>(d->a1); p.a1_ps = d->a1_pix_stride; p.c1 = d->c1;
  p.nimg = d->nimg; p.h = d->h; p.w = d->w; p.taps = d->taps;
  p.in_rows = d->in_rows > 0 ? d->in_rows : d->h; p.in_row0 = d->in_row0;
  for (int t = 0; t < 9; ++t) { p.tdy[t] = 0; p.tdx[t] = 0; }
  if (d->taps == 9) {
    for (int t = 0; t < 9; ++t) { p.tdy[t] = (signed char)(t / 3 - 1); p.tdx[t] = (signed char)(t % 3 - 1); }
  } else if (d->taps == 4) {
    const int a = d->tap_phase >> 1, b = d->tap_phase & 1;
    for (int t = 0; t < 4; ++t) { p.tdy[t] = (signed char)((t >> 1) - 1 + a); p.tdx[t] = (signed char)((t & 1) - 1 + b); }
  }
  p.wgt = reinterpret_cast<const float*>(d->wgt);
  p.ldw = d->ldw > 0 ? d->ldw : (long long)d->taps * (d->c0 + d->c1);
  p.n = d->n;
  p.out = d->out; p.ldo = d->ldo;
  p.osx = d->out_x_stride > 0 ? d->out_x_stride : d->ldo;
  p.osy = d->out_y_stride > 0 ? d->out_y_stride : p.osx * d->w;
  p.osi = d->out_img_stride > 0 ? d->out_img_stride : p.osy * d->h;
  p.bias = d->bias; p.rowadd = d->rowadd; p.ld_rowadd = d->ld_rowadd;
  p.residual = reinterpret_cast<const float*>(d->residual); p.ldr = d->ldr;
  p.mode = d->mode; p.alpha = d->alpha == 0.0f ? 1.0f : d->alpha;
  const long long M = (long long)d->nimg * d->h * d->w;
  dim3 grid((unsigned)((M + FT - 1) / FT), (unsigned)((d->n + FT - 1) / FT));
  f32_gemm_kernel<<<grid, 256, 0, STREAM>>>(p);
  return check_launch("igemm_f32");
}

extern "C" int dl_groupnorm_f32(const float* x0, int c0, const float* x1, int c1, int nimg, int hw, int groups,
                                float eps, const float* gamma, const float* beta, int apply_silu, float* out,
                                void* stream_) {
  DL_CHECK_ARG(x0 && out && gamma && beta && groups > 0 && (c0 + c1) % groups == 0 && (c1 == 0 || x1),
               "groupnorm_f32: bad args");
  f32_groupnorm_kernel<<<dim3(groups, nimg), 256, 0, STREAM>>>(x0, c0, x1, c1, hw, groups, eps, gamma, beta,
                                                              apply_silu, out);
  return check_launch("groupnorm_f32");
}

extern "C" int dl_layernorm_f32(const float* x, long long rows, int c, float eps, const float* gamma,
                                const float* beta, float* out, void* stream_) {
  DL_CHECK_ARG(x && out && gamma && beta && c > 0, "layernorm_f32: bad args");
  f32_layernorm_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, STREAM>>>(x, rows, c, eps, gamma, beta, out);
  return check_launch("layernorm_f32");
}

extern "C" int dl_attention_f32(const float* q, long long ldq, const float* k, long long ldk, const float* v,
                                long long ldv, int dh_stride, float* out, long long ldo, int batch, int sq,
                                int skv, int heads, int d, float scale, int causal, void* stream_) {
  DL_CHECK_ARG(q && k && v && out && d > 0 && d <= FA_MAXD, "attention_f32: bad args (d=%d)", d);
  const size_t smem = (size_t)(2 * FA_KEYS * (d + 1) + FA_WARPS * d) * sizeof(float);
  static bool attr_set[64] = {false};
  int dev = 0;
  cudaGetDevice(&dev);
  if (!attr_set[dev & 63]) {
    cudaFuncSetAttribute(f32_attention_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    attr_set[dev & 63] = true;
  }
  dim3 grid((sq + FA_WARPS - 1) / FA_WARPS, heads, batch);
  f32_attention_kernel<<<grid, FA_WARPS * 32, smem, STREAM>>>(q, ldq, k, ldk, v, ldv, dh_stride, out, ldo, sq, skv,
                                                             d, scale, causal);
  return check_launch("attention_f32");
}

extern "C" int dl_pack_latent_f32(const float* x, long long npix, int cin, int cpad, float scale,
                                  const float* mat, const float* vec, float* out, void* stream_) {
  DL_CHECK_ARG(x && out && cin <= cpad, "pack_latent_f32: bad args");
  f32_pack_latent_kernel<<<f32_grid(npix * cpad, 256), 256, 0, STREAM>>>(x, npix, cin, cpad, scale, mat, vec, out);
  return check_launch("pack_latent_f32");
}

extern "C" int dl_im2col_s2_f32(const float* x, int nimg, int h, int w, int c, float* cols, void* stream_) {
  DL_CHECK_ARG(x && cols && c % 4 == 0 && h % 2 == 0 && w % 2 == 0, "im2col_s2_f32: bad args");
  const long long total = (long long)nimg * (h / 2) * (w / 2) * 9 * (c / 4);
  f32_im2col_s2_kernel<<<f32_grid(total, 256), 256, 0, STREAM>>>(reinterpret_cast<const float4*>(x), nimg, h, w,
                                                                c / 4, reinterpret_cast<float4*>(cols), 1);
  return check_launch("im2col_s2_f32");
}

extern "C" int dl_im2col_s2_pad01_f32(const float* x, int nimg, int h, int w, int c, float* cols, void* stream_) {
  DL_CHECK_ARG(x && cols && c % 4 == 0 && h % 2 == 0 && w % 2 == 0, "im2col_s2_pad01_f32: bad args");
  const long long total = (long long)nimg * (h / 2) * (w / 2) * 9 * (c / 4);
  f32_im2col_s2_kernel<<<f32_grid(total, 256), 256, 0, STREAM>>>(reinterpret_cast<const float4*>(x), nimg, h, w,
                                                                c / 4, reinterpret_cast<float4*>(cols), 0);
  return check_launch("im2col_s2_pad01_f32");
}

extern "C" int dl_softmax_rows_f32(const float* scores, long long rows, int cols, float* out, void* stream_) {
  DL_CHECK_ARG(scores && out && rows > 0 && cols > 0, "softmax_rows_f32: bad args");
  f32_softmax_rows_kernel<<<(unsigned)rows, 256, 0, STREAM>>>(scores, rows, cols, out);
  return check_launch("softmax_rows_f32");
}

extern "C" int dl_small_linear_f32(const float* x, int m, int k, const float* w, const float* bias,
                                   const float* add, int n, int silu_in, int silu_out, float* out,
                                   void* stream_) {
  DL_CHECK_ARG(x && w && out && m >= 1 && n >= 1, "small_linear_f32: bad args");
  const long long warps = (long long)n * m;
  f32_small_linear_kernel<<<(unsigned)((warps * 32 + 255) / 256), 256, 0, STREAM>>>(x, m, k, w, bias, add, n,
                                                                                   silu_in, silu_out, out);
  return check_launch("small_linear_f32");
}
