// Bandwidth-/latency-bound pieces of the hot path (SURVEY.md K9-K11, K15): timestep embedding,
// tiny time-MLP GEMMs, nearest-2x upsample, stride-2 im2col, latent packing, the fused LCM
// scheduler update and the 8x8 latent pool.  All vectorised (16-byte) and coalesced.
#include <cuda_fp16.h>

#include "common.cuh"
#include "dreamlab_b200.h"

namespace dl {

// ---- Timesteps(dim, flip_sin_to_cos=True, freq_shift=0) ---------------------------------------
__global__ void sinusoid_kernel(const float* __restrict__ t, int batch, int dim,
                                float* __restrict__ out) {
  const int half = dim / 2;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= batch * half) return;
  const int b = i / half, k = i % half;
  // exp(-ln(10000) * k / half) in fp32, then t * f: same op order as the oracle
  const float f = expf(-9.210340371976184f * (float)k / (float)half);
  const float a = t[b] * f;
  out[(size_t)b * dim + k] = cosf(a);
  out[(size_t)b * dim + half + k] = sinf(a);
}

// ---- out[m,n] = act_out(sum_k act_in(x[m,k]) w[n,k] + bias[n] + add[m,n]) --------------------
// One warp per NR consecutive output columns: the x chunk a lane loads (MMAX rows x 8 values) is
// reused for NR weight rows, so the L1 traffic for x — 30x the weight bytes with one column per
// warp — drops NR-fold; act_in is applied once per loaded value, not once per output column.
template <int MMAX, int NR>
__global__ void small_linear_kernel(const float* __restrict__ x, int m, int k,
                                    const __nv_bfloat16* __restrict__ w,
                                    const float* __restrict__ bias, const float* __restrict__ add,
                                    int n, int silu_in, int silu_out, float* __restrict__ out) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  const int n0 = warp * NR;
  if (n0 >= n) return;
  float acc[NR][MMAX];
#pragma unroll
  for (int r = 0; r < NR; ++r)
#pragma unroll
    for (int i = 0; i < MMAX; ++i) acc[r][i] = 0.f;
  for (int kk = lane * 8; kk < k; kk += 256) {
    float wf[NR][8];
#pragma unroll
    for (int r = 0; r < NR; ++r) {
      const int row = min(n0 + r, n - 1);
      const uint4 u = __ldg(reinterpret_cast<const uint4*>(w + (size_t)row * k + kk));
      const uint32_t ww[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float2 f = unpack_bf16x2(ww[j]);
        wf[r][2 * j] = f.x; wf[r][2 * j + 1] = f.y;
      }
    }
#pragma unroll
    for (int i = 0; i < MMAX; ++i) {
      if (i < m) {
        const float4 a0 = __ldg(reinterpret_cast<const float4*>(x + (size_t)i * k + kk));
        const float4 a1 = __ldg(reinterpret_cast<const float4*>(x + (size_t)i * k + kk + 4));
        float xv[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
        if (silu_in) {
#pragma unroll
          for (int j = 0; j < 8; ++j) xv[j] = silu_f(xv[j]);
        }
#pragma unroll
        for (int r = 0; r < NR; ++r)
#pragma unroll
          for (int j = 0; j < 8; ++j) acc[r][i] += xv[j] * wf[r][j];
      }
    }
  }
#pragma unroll
  for (int r = 0; r < NR; ++r) {
    const int col = n0 + r;
#pragma unroll
    for (int i = 0; i < MMAX; ++i) {
      const float s = warp_sum(acc[r][i]);
      if (lane == 0 && i < m && col < n) {
        float v = s + (bias ? bias[col] : 0.f) + (add ? add[(size_t)i * n + col] : 0.f);
        if (silu_out) v = silu_f(v);
        out[(size_t)i * n + col] = v;
      }
    }
  }
}

// ---- nearest 2x upsample, NHWC bf16 ---------------------------------------------------------
__global__ void upsample2x_kernel(const uint4* __restrict__ x, int nimg, int h, int w, int V,
                                  uint4* __restrict__ out) {
  const long long total = (long long)nimg * h * w * V;   // one thread per input vector
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int v = (int)(i % V);
    long long p = i / V;
    const int xx = (int)(p % w);
    p /= w;
    const int yy = (int)(p % h);
    const int n = (int)(p / h);
    const uint4 val = __ldg(x + i);
    const long long ow = 2LL * w;
    const long long base = (((long long)n * 2 * h + 2 * yy) * ow + 2 * xx) * V + v;
    out[base] = val;
    out[base + V] = val;
    out[base + ow * V] = val;
    out[base + ow * V + V] = val;
  }
}

// ---- im2col for conv3x3 stride 2 (Downsample2D): cols[(n,yo,xo), tap*c + ch] -----------------
// pad = 1: the UNet's symmetric padding 1; pad = 0: the VAE encoder's F.pad(x, (0,1,0,1)) followed
// by an unpadded conv (tap (ky,kx) of output (yo,xo) reads input (2yo+ky, 2xo+kx), the last row and
// column of taps fall on the zero pad)
__global__ void im2col_s2_kernel(const uint4* __restrict__ x, int nimg, int h, int w, int V,
                                 uint4* __restrict__ cols, int in_rows, int in_row0, int pad) {
  const int ho = h / 2, wo = w / 2;
  const long long total = (long long)nimg * ho * wo * 9 * V;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int v = (int)(i % V);
    long long r = i / V;
    const int tap = (int)(r % 9);
    r /= 9;
    const int xo = (int)(r % wo);
    r /= wo;
    const int yo = (int)(r % ho);
    const int n = (int)(r / ho);
    const int yi = 2 * yo + tap / 3 - pad + in_row0;
    const int xi = 2 * xo + tap % 3 - pad;
    uint4 val = make_uint4(0, 0, 0, 0);
    if (yi >= 0 && yi < in_rows && xi >= 0 && xi < w)
      val = __ldg(x + (((long long)n * in_rows + yi) * w + xi) * V + v);
    cols[i] = val;
  }
}

// out[p, c] = bf16( sum_j mat[c][j] * (x[p, j] * scale) + vec[c] ) for c < cin, 0 for the pad
// (mat == NULL: identity).  The optional cin x cin matrix is the VAE post_quant_conv (1x1).
__global__ void pack_latent_kernel(const float* __restrict__ x, long long npix, int cin, int cpad,
                                   float scale, const float* __restrict__ mat,
                                   const float* __restrict__ vec, __nv_bfloat16* __restrict__ out) {
  const long long total = npix * cpad;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(i % cpad);
    const long long p = i / cpad;
    float r = 0.f;
    if (c < cin) {
      if (mat == nullptr) {
        r = x[p * cin + c] * scale;
      } else {
        r = vec ? vec[c] : 0.f;
        for (int j = 0; j < cin; ++j) r += mat[c * cin + j] * (x[p * cin + j] * scale);
      }
    }
    out[i] = __float2bfloat16(r);
  }
}

// row softmax: fp32 scores [rows, cols] -> bf16 probabilities (VAE mid-block attention, d=512)
__global__ void softmax_rows_kernel(const float* __restrict__ s, long long rows, int cols,
                                    __nv_bfloat16* __restrict__ out) {
  __shared__ float red[32];
  const long long row = blockIdx.x;
  const float* sr = s + row * cols;
  float m = -INFINITY;
  for (int i = threadIdx.x; i < cols; i += blockDim.x) m = fmaxf(m, sr[i]);
  m = warp_max(m);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x < 32) {
    float v = threadIdx.x < (blockDim.x >> 5) ? red[threadIdx.x] : -INFINITY;
    v = warp_max(v);
    if (threadIdx.x == 0) red[0] = v;
  }
  __syncthreads();
  m = red[0];
  __syncthreads();
  float l = 0.f;
  for (int i = threadIdx.x; i < cols; i += blockDim.x) l += __expf(sr[i] - m);
  l = warp_sum(l);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = l;
  __syncthreads();
  if (threadIdx.x < 32) {
    float v = threadIdx.x < (blockDim.x >> 5) ? red[threadIdx.x] : 0.f;
    v = warp_sum(v);
    if (threadIdx.x == 0) red[0] = v;
  }
  __syncthreads();
  const float inv = 1.f / red[0];
  for (int i = threadIdx.x; i < cols; i += blockDim.x)
    out[row * cols + i] = __float2bfloat16(__expf(sr[i] - m) * inv);
}

__global__ void nchw_to_nhwc_kernel(const float* __restrict__ x, int nimg, int c, int hw,
                                    float* __restrict__ out) {
  const long long total = (long long)nimg * c * hw;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int ch = (int)(i % c);
    long long r = i / c;
    const int p = (int)(r % hw);
    const int n = (int)(r / hw);
    out[i] = x[((long long)n * c + ch) * hw + p];
  }
}
__global__ void nhwc_to_nchw_kernel(const float* __restrict__ x, int nimg, int c, int hw,
                                    float* __restrict__ out) {
  const long long total = (long long)nimg * c * hw;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int p = (int)(i % hw);
    long long r = i / hw;
    const int ch = (int)(r % c);
    const int n = (int)(r / c);
    out[i] = x[((long long)n * hw + p) * c + ch];
  }
}

// ---- LCMScheduler.step, fused (fp32 latents; coefficients are the scheduler's fp32 scalars) ---
// PRED (DL_PRED_*) picks how x0 follows from the model output (lcm_x0 in common.cuh); clip: clamp x0 to [-r, r].
template <int PRED>
__global__ void lcm_step_kernel(const float4* __restrict__ eps, const float4* __restrict__ x,
                                const float4* __restrict__ noise, float4* __restrict__ x_next,
                                float4* __restrict__ denoised, long long n4, dl_lcm_coeffs k, int clip, float r) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4;
       i += (long long)gridDim.x * blockDim.x) {
    const float4 e = eps[i], xv = x[i];
    const float ev[4] = {e.x, e.y, e.z, e.w};
    const float xx[4] = {xv.x, xv.y, xv.z, xv.w};
    float zz[4] = {0.f, 0.f, 0.f, 0.f};
    if (noise != nullptr) {
      const float4 z = noise[i];
      zz[0] = z.x; zz[1] = z.y; zz[2] = z.z; zz[3] = z.w;
    }
    float d[4], o[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      // no FMA contraction: keep the reference's op order (x0, then mul, mul, add)
      const float x0 = lcm_x0<PRED>(ev[j], xx[j], k.sqrt_alpha_t, k.sqrt_beta_t, clip, r);
      d[j] = __fadd_rn(__fmul_rn(k.c_out, x0), __fmul_rn(k.c_skip, xx[j]));
      o[j] = (noise != nullptr)
                 ? __fadd_rn(__fmul_rn(k.sqrt_alpha_prev, d[j]), __fmul_rn(k.sqrt_beta_prev, zz[j]))
                 : d[j];
    }
    denoised[i] = make_float4(d[0], d[1], d[2], d[3]);
    x_next[i] = make_float4(o[0], o[1], o[2], o[3]);
  }
}

// ---- CLIP text tower pieces (transformers CLIPTextModel: embeddings, MLP activation) -----------
// out[i, :] = bf16( tok[ids[i], :] + pos[i % seq, :] ), 8 channels per thread
__global__ void embed_tokens_kernel(const long long* __restrict__ ids, const __nv_bfloat16* __restrict__ tok,
                                    const __nv_bfloat16* __restrict__ pos, int n, int seq, int vocab, int V,
                                    uint4* __restrict__ out) {
  const long long total = (long long)n * V;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int v = (int)(i % V);
    const int r = (int)(i / V);
    long long id = ids[r];
    id = id < 0 ? 0 : (id >= vocab ? vocab - 1 : id);
    const uint4 a = __ldg(reinterpret_cast<const uint4*>(tok + id * (long long)V * 8) + v);
    const uint4 b = __ldg(reinterpret_cast<const uint4*>(pos + (long long)(r % seq) * V * 8) + v);
    const uint32_t aw[4] = {a.x, a.y, a.z, a.w}, bw[4] = {b.x, b.y, b.z, b.w};
    uint32_t o[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float2 fa = unpack_bf16x2(aw[j]), fb = unpack_bf16x2(bw[j]);
      o[j] = pack_bf16x2(fa.x + fb.x, fa.y + fb.y);
    }
    out[i] = make_uint4(o[0], o[1], o[2], o[3]);
  }
}

// mode 0: quick_gelu x * sigmoid(1.702 x) (CLIP-L);  mode 1: exact (erf) GELU (OpenCLIP bigG)
__global__ void act_bf16_kernel(const uint4* __restrict__ x, uint4* __restrict__ out, long long n8, int mode) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n8;
       i += (long long)gridDim.x * blockDim.x) {
    const uint4 u = x[i];
    const uint32_t w[4] = {u.x, u.y, u.z, u.w};
    uint32_t o[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float2 f = unpack_bf16x2(w[j]);
      if (mode == 0) {
        f.x = f.x / (1.0f + __expf(-1.702f * f.x));
        f.y = f.y / (1.0f + __expf(-1.702f * f.y));
      } else {
        f.x = 0.5f * f.x * (1.0f + erff(f.x * 0.70710678118654752f));
        f.y = 0.5f * f.y * (1.0f + erff(f.y * 0.70710678118654752f));
      }
      o[j] = pack_bf16x2(f.x, f.y);
    }
    out[i] = make_uint4(o[0], o[1], o[2], o[3]);
  }
}

// ---- tiled VAE decode (diffusers AutoencoderKL.tiled_decode: blend_v / blend_h / crop) ----------
// b[n, y, x, :] (y < extent) = a[n, ha - extent + y, x, :] * (1 - y/extent) + b[n, y, x, :] * (y/extent)
// vertical = 1 blends along rows (a above b, same width), 0 along columns (a left of b, same height)
__global__ void tile_blend_kernel(const float* __restrict__ a, float* __restrict__ b, int nimg, int ha,
                                  int wa, int hb, int wb, int c, int extent, int vertical) {
  const int bh = vertical ? extent : hb, bw = vertical ? wb : extent;
  const long long total = (long long)nimg * bh * bw * c;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int ch = (int)(i % c);
    long long r = i / c;
    const int x = (int)(r % bw);
    r /= bw;
    const int y = (int)(r % bh);
    const int n = (int)(r / bh);
    const int k = vertical ? y : x;
    const float wb_ = (float)((double)k / (double)extent);
    const float wa_ = (float)(1.0 - (double)k / (double)extent);
    const long long ia = vertical ? (((long long)n * ha + (ha - extent + y)) * wa + x) * c + ch
                                  : (((long long)n * ha + y) * wa + (wa - extent + x)) * c + ch;
    const long long ib = (((long long)n * hb + y) * wb + x) * c + ch;
    b[ib] = __fadd_rn(__fmul_rn(a[ia], wa_), __fmul_rn(b[ib], wb_));
  }
}

// crop [0,ch) x [0,cw) of an fp32 NHWC image tile -> u8 canvas window with the VaeImageProcessor
// tail of the untiled path (bf16-rounded decoder output, clamp(x/2+0.5,0,1)*255, round-half-even)
__global__ void image_crop_u8_kernel(const float* __restrict__ src, int nimg, int hs, int ws, int c,
                                     int ch, int cw, uint8_t* __restrict__ dst, long long dst_row_stride,
                                     long long dst_img_stride) {
  const long long total = (long long)nimg * ch * cw * c;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int k = (int)(i % c);
    long long r = i / c;
    const int x = (int)(r % cw);
    r /= cw;
    const int y = (int)(r % ch);
    const int n = (int)(r / ch);
    const float v = src[(((long long)n * hs + y) * ws + x) * c + k];
    const float xb = __bfloat162float(__float2bfloat16(v));
    const float f = fminf(fmaxf(xb * 0.5f + 0.5f, 0.0f), 1.0f) * 255.0f;
    dst[(long long)n * dst_img_stride + (long long)y * dst_row_stride + (long long)x * c + k] =
        (uint8_t)__float2int_rn(f);
  }
}

// ---- classifier-free guidance: out = u + gs * (t - u), un-contracted like the reference ------
__global__ void cfg_combine_kernel(const float4* __restrict__ u, const float4* __restrict__ t, float gs,
                                   float4* __restrict__ out, long long n4) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n4;
       i += (long long)gridDim.x * blockDim.x) {
    const float4 a = u[i], b = t[i];
    float4 o;
    o.x = __fadd_rn(a.x, __fmul_rn(gs, __fsub_rn(b.x, a.x)));
    o.y = __fadd_rn(a.y, __fmul_rn(gs, __fsub_rn(b.y, a.y)));
    o.z = __fadd_rn(a.z, __fmul_rn(gs, __fsub_rn(b.z, a.z)));
    o.w = __fadd_rn(a.w, __fmul_rn(gs, __fsub_rn(b.w, a.w)));
    out[i] = o;
  }
}

// ---- sampler step (Euler, Euler ancestral, DDIM, DPM++ 2M): guidance + one linear form, fused ----------------
// e = u + gs (t - u) (cfg_combine's roundings; t == null: e = u);  x0 = clamp(a_x x + a_e e);
// x_next = c_x x + c_e e + c_0 x0 + c_1 x0_prev + c_n z, every mul / add rounded on its own, summed left to right
__global__ void sampler_step_kernel(const float4* __restrict__ u, const float4* __restrict__ t, float gs,
                                    const float4* __restrict__ x, const float4* __restrict__ x0_prev,
                                    const float4* __restrict__ noise, float4* __restrict__ x_next,
                                    float4* __restrict__ x0_out, long long n4, dl_sampler_coeffs k) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4;
       i += (long long)gridDim.x * blockDim.x) {
    const float4 uv = u[i], xv = x[i];
    float e[4] = {uv.x, uv.y, uv.z, uv.w};
    const float xx[4] = {xv.x, xv.y, xv.z, xv.w};
    if (t != nullptr) {
      const float4 tv = t[i];
      const float tt[4] = {tv.x, tv.y, tv.z, tv.w};
#pragma unroll
      for (int j = 0; j < 4; ++j) e[j] = __fadd_rn(e[j], __fmul_rn(gs, __fsub_rn(tt[j], e[j])));
    }
    float pp[4] = {0.f, 0.f, 0.f, 0.f}, zz[4] = {0.f, 0.f, 0.f, 0.f};
    if (x0_prev != nullptr) {
      const float4 p = x0_prev[i];
      pp[0] = p.x; pp[1] = p.y; pp[2] = p.z; pp[3] = p.w;
    }
    if (noise != nullptr) {
      const float4 z = noise[i];
      zz[0] = z.x; zz[1] = z.y; zz[2] = z.z; zz[3] = z.w;
    }
    float d[4], o[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float x0 = __fadd_rn(__fmul_rn(k.a_x, xx[j]), __fmul_rn(k.a_e, e[j]));
      if (k.clip_sample) x0 = fminf(fmaxf(x0, -k.clip_sample_range), k.clip_sample_range);
      float v = __fadd_rn(__fmul_rn(k.c_x, xx[j]), __fmul_rn(k.c_e, e[j]));
      v = __fadd_rn(v, __fmul_rn(k.c_0, x0));
      if (x0_prev != nullptr) v = __fadd_rn(v, __fmul_rn(k.c_1, pp[j]));
      if (noise != nullptr) v = __fadd_rn(v, __fmul_rn(k.c_n, zz[j]));
      d[j] = x0;
      o[j] = v;
    }
    x0_out[i] = make_float4(d[0], d[1], d[2], d[3]);
    x_next[i] = make_float4(o[0], o[1], o[2], o[3]);
  }
}

// ---- fp32 adaptive_avg_pool2d -> (8,8) -> fp16, NHWC in, NCHW out -----------------------------
__global__ void latent_pool8_kernel(const float* __restrict__ lat, int nimg, int h, int w, int c,
                                    __half* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nimg * c * 64) return;
  const int ox = i % 8, oy = (i / 8) % 8, ch = (i / 64) % c, n = i / (64 * c);
  // torch.nn.functional.adaptive_avg_pool2d bins: [floor(i*H/8), ceil((i+1)*H/8)) — equal blocks when
  // H, W are multiples of 8 (reference `backends/cuda_worker.py:299`), overlapping bins otherwise
  const int y0 = (oy * h) / 8, y1 = ((oy + 1) * h + 7) / 8;
  const int x0 = (ox * w) / 8, x1 = ((ox + 1) * w + 7) / 8;
  float s = 0.f;
  for (int y = y0; y < y1; ++y)
    for (int x = x0; x < x1; ++x)
      s += lat[(((long long)n * h + y) * w + x) * c + ch];
  out[i] = __float2half_rn(s / (float)((y1 - y0) * (x1 - x0)));
}

// ---- narrow-output conv3x3 as a 1x1 GEMM + tap sum (VAE conv_out, 128 -> 3 channels) -----------------------
// A 3x3 conv with 3 output channels wastes the tensor core (N = 16 tile at 2 % of peak) and re-reads its 1 GB
// input nine times through the TMA pipeline.  Instead ONE 1x1 GEMM computes, per INPUT pixel q, the 27 partial
// products Y[q, t, oc] = w[oc, tap t, :] . in[q, :] (input read once), and this kernel gathers
//   out[p, oc] = bias[oc] + sum_t Y[p + offset(t), t, oc]          (zero padding: out-of-image taps skipped)
// and applies the VaeImageProcessor tail (reference `backends/rknnlcm.py:220-235`) when the output is u8.
template <bool U8>
__global__ void conv_tapsum_kernel(const float* __restrict__ yp, int nimg, int h, int w, int ldy, int nout,
                                   const float* __restrict__ bias, void* __restrict__ out) {
  const long long total = (long long)nimg * h * w;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int x = (int)(i % w);
    const int y = (int)((i / w) % h);
    float acc[4];
#pragma unroll
    for (int oc = 0; oc < 4; ++oc) acc[oc] = oc < nout ? __ldg(bias + oc) : 0.f;
#pragma unroll
    for (int t = 0; t < 9; ++t) {
      const int yy = y + t / 3 - 1, xx = x + t % 3 - 1;
      if (yy < 0 || yy >= h || xx < 0 || xx >= w) continue;
      const float* q = yp + (i + (long long)(t / 3 - 1) * w + (t % 3 - 1)) * ldy + t * nout;
#pragma unroll
      for (int oc = 0; oc < 4; ++oc)
        if (oc < nout) acc[oc] += __ldg(q + oc);
    }
    if (U8) {
      uint8_t* o = reinterpret_cast<uint8_t*>(out) + i * nout;
#pragma unroll
      for (int oc = 0; oc < 4; ++oc)
        if (oc < nout) {
          const float xb = __bfloat162float(__float2bfloat16(acc[oc]));   // the decoder's output dtype
          o[oc] = (uint8_t)__float2int_rn(fminf(fmaxf(xb * 0.5f + 0.5f, 0.0f), 1.0f) * 255.0f);
        }
    } else {
      float* o = reinterpret_cast<float*>(out) + i * nout;
#pragma unroll
      for (int oc = 0; oc < 4; ++oc)
        if (oc < nout) o[oc] = acc[oc];
    }
  }
}

static inline unsigned grid_for(long long total, int threads) {
  long long b = (total + threads - 1) / threads;
  const long long cap = (long long)num_sms() * 16;
  if (b > cap) b = cap;
  if (b < 1) b = 1;
  return (unsigned)b;
}

}  // namespace dl

using namespace dl;
#define STREAM reinterpret_cast<cudaStream_t>(stream_)

extern "C" int dl_timestep_sinusoid(const float* t, int batch, int dim, float* out, void* stream_) {
  DL_CHECK_ARG(t && out && dim % 2 == 0 && batch > 0, "timestep_sinusoid: bad args");
  const int total = batch * dim / 2;
  sinusoid_kernel<<<(total + 127) / 128, 128, 0, STREAM>>>(t, batch, dim, out);
  return check_launch("timestep_sinusoid");
}

extern "C" int dl_small_linear(const float* x, int m, int k, const void* w, const float* bias,
                               const float* add, int n, int silu_in, int silu_out, float* out,
                               void* stream_) {
  DL_CHECK_ARG(x && w && out, "small_linear: null pointer");
  DL_CHECK_ARG(k % 8 == 0, "small_linear: k=%d must be a multiple of 8", k);
  DL_CHECK_ARG(m >= 1 && m <= 64, "small_linear: m=%d must be in [1,64]", m);
  const int threads = 256;
  // wide outputs (the fused time_emb_proj matrix): 4 columns per warp share the x chunk; narrow
  // ones (time MLP): one column per warp so that the few hundred outputs still fill the SMs
  const int nr = n >= 8192 ? 4 : 1;
  const int blocks = (((n + nr - 1) / nr) * 32 + threads - 1) / threads;
  const __nv_bfloat16* wb = reinterpret_cast<const __nv_bfloat16*>(w);
  for (int m0 = 0; m0 < m; m0 += 16) {
    const int mm = (m - m0) < 16 ? (m - m0) : 16;
    if (nr == 4)
      small_linear_kernel<16, 4><<<blocks, threads, 0, STREAM>>>(
          x + (size_t)m0 * k, mm, k, wb, bias, add ? add + (size_t)m0 * n : nullptr, n, silu_in,
          silu_out, out + (size_t)m0 * n);
    else
      small_linear_kernel<16, 1><<<blocks, threads, 0, STREAM>>>(
          x + (size_t)m0 * k, mm, k, wb, bias, add ? add + (size_t)m0 * n : nullptr, n, silu_in,
          silu_out, out + (size_t)m0 * n);
  }
  return check_launch("small_linear");
}

extern "C" int dl_upsample2x(const void* x, int nimg, int h, int w, int c, void* out, void* stream_) {
  DL_CHECK_ARG(x && out && c % 8 == 0, "upsample2x: bad args");
  const long long total = (long long)nimg * h * w * (c / 8);
  upsample2x_kernel<<<grid_for(total, 256), 256, 0, STREAM>>>(
      reinterpret_cast<const uint4*>(x), nimg, h, w, c / 8, reinterpret_cast<uint4*>(out));
  return check_launch("upsample2x");
}

extern "C" int dl_im2col_s2(const void* x, int nimg, int h, int w, int c, void* cols, void* stream_) {
  DL_CHECK_ARG(x && cols && c % 8 == 0 && h % 2 == 0 && w % 2 == 0, "im2col_s2: bad args");
  const long long total = (long long)nimg * (h / 2) * (w / 2) * 9 * (c / 8);
  im2col_s2_kernel<<<grid_for(total, 256), 256, 0, STREAM>>>(
      reinterpret_cast<const uint4*>(x), nimg, h, w, c / 8, reinterpret_cast<uint4*>(cols), h, 0, 1);
  return check_launch("im2col_s2");
}

extern "C" int dl_im2col_s2_pad01(const void* x, int nimg, int h, int w, int c, void* cols, void* stream_) {
  DL_CHECK_ARG(x && cols && c % 8 == 0 && h % 2 == 0 && w % 2 == 0, "im2col_s2_pad01: bad args");
  const long long total = (long long)nimg * (h / 2) * (w / 2) * 9 * (c / 8);
  im2col_s2_kernel<<<grid_for(total, 256), 256, 0, STREAM>>>(
      reinterpret_cast<const uint4*>(x), nimg, h, w, c / 8, reinterpret_cast<uint4*>(cols), h, 0, 0);
  return check_launch("im2col_s2_pad01");
}

extern "C" int dl_im2col_s2_halo(const void* x, int nimg, int in_rows, int in_row0, int h, int w, int c,
                                 void* cols, void* stream_) {
  DL_CHECK_ARG(x && cols && c % 8 == 0 && h % 2 == 0 && w % 2 == 0 && in_rows >= h && in_row0 >= 0,
               "im2col_s2_halo: bad args");
  const long long total = (long long)nimg * (h / 2) * (w / 2) * 9 * (c / 8);
  im2col_s2_kernel<<<grid_for(total, 256), 256, 0, STREAM>>>(
      reinterpret_cast<const uint4*>(x), nimg, h, w, c / 8, reinterpret_cast<uint4*>(cols), in_rows, in_row0, 1);
  return check_launch("im2col_s2_halo");
}

extern "C" int dl_pack_latent(const float* x, long long npix, int cin, int cpad, float scale,
                              const float* mat, const float* vec, void* out, void* stream_) {
  DL_CHECK_ARG(x && out && cin <= cpad, "pack_latent: bad args");
  pack_latent_kernel<<<grid_for(npix * cpad, 256), 256, 0, STREAM>>>(
      x, npix, cin, cpad, scale, mat, vec, reinterpret_cast<__nv_bfloat16*>(out));
  return check_launch("pack_latent");
}

namespace dl {
// same, row held in registers (cols <= 256 * 16, cols % 4 == 0): one read of the scores instead of
// three, float4 loads, packed 8-byte bf16 stores
__global__ void __launch_bounds__(256) softmax_rows_reg_kernel(const float* __restrict__ s, long long rows, int cols,
                                                               __nv_bfloat16* __restrict__ out) {
  __shared__ float red[8];
  const long long row = blockIdx.x;
  const float4* sr = reinterpret_cast<const float4*>(s + row * cols);
  const int n4 = cols >> 2;
  float4 v[4];
  float m = -INFINITY;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int i = threadIdx.x + j * 256;
    v[j] = i < n4 ? __ldg(sr + i) : make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
    m = fmaxf(m, fmaxf(fmaxf(v[j].x, v[j].y), fmaxf(v[j].z, v[j].w)));
  }
  m = warp_max(m);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
  __syncthreads();
  m = red[0];
#pragma unroll
  for (int w = 1; w < 8; ++w) m = fmaxf(m, red[w]);
  __syncthreads();
  float l = 0.f;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    v[j].x = __expf(v[j].x - m); v[j].y = __expf(v[j].y - m);
    v[j].z = __expf(v[j].z - m); v[j].w = __expf(v[j].w - m);
    l += (v[j].x + v[j].y) + (v[j].z + v[j].w);
  }
  l = warp_sum(l);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = l;
  __syncthreads();
  float tot = 0.f;
#pragma unroll
  for (int w = 0; w < 8; ++w) tot += red[w];
  const float inv = 1.f / tot;
  uint2* orow = reinterpret_cast<uint2*>(out + row * cols);
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int i = threadIdx.x + j * 256;
    if (i < n4) orow[i] = make_uint2(pack_bf16x2(v[j].x * inv, v[j].y * inv), pack_bf16x2(v[j].z * inv, v[j].w * inv));
  }
}
}  // namespace dl

extern "C" int dl_softmax_rows(const float* scores, long long rows, int cols, void* out,
                               void* stream_) {
  DL_CHECK_ARG(scores && out && rows > 0 && cols > 0, "softmax_rows: bad args");
  if (cols % 4 == 0 && cols <= 4096)
    softmax_rows_reg_kernel<<<(unsigned)rows, 256, 0, STREAM>>>(scores, rows, cols,
                                                               reinterpret_cast<__nv_bfloat16*>(out));
  else
    softmax_rows_kernel<<<(unsigned)rows, 256, 0, STREAM>>>(scores, rows, cols,
                                                           reinterpret_cast<__nv_bfloat16*>(out));
  return check_launch("softmax_rows");
}

extern "C" int dl_nchw_to_nhwc_f32(const float* x, int nimg, int c, int hw, float* out, void* stream_) {
  DL_CHECK_ARG(x && out, "nchw_to_nhwc: null pointer");
  nchw_to_nhwc_kernel<<<grid_for((long long)nimg * c * hw, 256), 256, 0, STREAM>>>(x, nimg, c, hw, out);
  return check_launch("nchw_to_nhwc");
}
extern "C" int dl_nhwc_to_nchw_f32(const float* x, int nimg, int c, int hw, float* out, void* stream_) {
  DL_CHECK_ARG(x && out, "nhwc_to_nchw: null pointer");
  nhwc_to_nchw_kernel<<<grid_for((long long)nimg * c * hw, 256), 256, 0, STREAM>>>(x, nimg, c, hw, out);
  return check_launch("nhwc_to_nchw");
}

extern "C" int dl_lcm_step(const float* eps, const float* x, const float* noise, float* x_next,
                           float* denoised, long long n, const dl_lcm_coeffs* k, void* stream_) {
  DL_CHECK_ARG(eps && x && x_next && denoised && k, "lcm_step: null pointer");
  DL_CHECK_ARG(n % 4 == 0, "lcm_step: n must be a multiple of 4");
  lcm_step_kernel<DL_PRED_EPSILON><<<grid_for(n / 4, 256), 256, 0, STREAM>>>(
      reinterpret_cast<const float4*>(eps), reinterpret_cast<const float4*>(x),
      reinterpret_cast<const float4*>(noise), reinterpret_cast<float4*>(x_next),
      reinterpret_cast<float4*>(denoised), n / 4, *k, 0, 0.f);
  return check_launch("lcm_step");
}

extern "C" int dl_lcm_step_ex(const float* mo, const float* x, const float* noise, float* x_next,
                              float* denoised, long long n, const dl_lcm_coeffs_ex* k, void* stream_) {
  DL_CHECK_ARG(mo && x && x_next && denoised && k, "lcm_step_ex: null pointer");
  DL_CHECK_ARG(n % 4 == 0, "lcm_step_ex: n must be a multiple of 4");
  DL_CHECK_ARG(!k->clip_sample || k->clip_sample_range >= 0.f, "lcm_step_ex: clip_sample_range must be >= 0");
  const unsigned grid = grid_for(n / 4, 256);
  const float4* m4 = reinterpret_cast<const float4*>(mo);
  const float4* x4 = reinterpret_cast<const float4*>(x);
  const float4* z4 = reinterpret_cast<const float4*>(noise);
  float4* o4 = reinterpret_cast<float4*>(x_next);
  float4* d4 = reinterpret_cast<float4*>(denoised);
  const int clip = k->clip_sample != 0;
  switch (k->prediction_type) {
    case DL_PRED_EPSILON:
      lcm_step_kernel<DL_PRED_EPSILON><<<grid, 256, 0, STREAM>>>(m4, x4, z4, o4, d4, n / 4, k->k, clip,
                                                                  k->clip_sample_range);
      break;
    case DL_PRED_V:
      lcm_step_kernel<DL_PRED_V><<<grid, 256, 0, STREAM>>>(m4, x4, z4, o4, d4, n / 4, k->k, clip,
                                                            k->clip_sample_range);
      break;
    case DL_PRED_SAMPLE:
      lcm_step_kernel<DL_PRED_SAMPLE><<<grid, 256, 0, STREAM>>>(m4, x4, z4, o4, d4, n / 4, k->k, clip,
                                                                 k->clip_sample_range);
      break;
    default:
      DL_CHECK_ARG(false, "lcm_step_ex: unknown prediction_type");
  }
  return check_launch("lcm_step_ex");
}

extern "C" int dl_embed_tokens(const long long* ids, const void* tok_emb, const void* pos_emb, int n, int seq,
                               int vocab, int dim, void* out, void* stream_) {
  DL_CHECK_ARG(ids && tok_emb && pos_emb && out && n > 0 && seq > 0 && vocab > 0 && dim % 8 == 0,
               "embed_tokens: bad args");
  embed_tokens_kernel<<<grid_for((long long)n * (dim / 8), 256), 256, 0, STREAM>>>(
      ids, reinterpret_cast<const __nv_bfloat16*>(tok_emb), reinterpret_cast<const __nv_bfloat16*>(pos_emb), n, seq,
      vocab, dim / 8, reinterpret_cast<uint4*>(out));
  return check_launch("embed_tokens");
}

extern "C" int dl_act_bf16(const void* x, void* out, long long n, int mode, void* stream_) {
  DL_CHECK_ARG(x && out && n % 8 == 0 && (mode == 0 || mode == 1), "act_bf16: bad args");
  act_bf16_kernel<<<grid_for(n / 8, 256), 256, 0, STREAM>>>(reinterpret_cast<const uint4*>(x),
                                                           reinterpret_cast<uint4*>(out), n / 8, mode);
  return check_launch("act_bf16");
}

extern "C" int dl_tile_blend(const float* a, float* b, int nimg, int ha, int wa, int hb, int wb, int c,
                             int extent, int vertical, void* stream_) {
  DL_CHECK_ARG(a && b && nimg > 0 && c > 0 && extent > 0, "tile_blend: bad args");
  DL_CHECK_ARG(vertical ? (wa == wb && extent <= ha && extent <= hb) : (ha == hb && extent <= wa && extent <= wb),
               "tile_blend: tiles do not line up (a %dx%d, b %dx%d, extent %d)", ha, wa, hb, wb, extent);
  const long long total = (long long)nimg * (vertical ? extent : hb) * (vertical ? wb : extent) * c;
  tile_blend_kernel<<<grid_for(total, 256), 256, 0, STREAM>>>(a, b, nimg, ha, wa, hb, wb, c, extent, vertical);
  return check_launch("tile_blend");
}

extern "C" int dl_image_crop_u8(const float* src, int nimg, int hs, int ws, int c, int crop_h, int crop_w,
                                void* dst_u8, long long dst_row_stride, long long dst_img_stride,
                                void* stream_) {
  DL_CHECK_ARG(src && dst_u8 && crop_h > 0 && crop_w > 0 && crop_h <= hs && crop_w <= ws, "image_crop_u8: bad args");
  const long long total = (long long)nimg * crop_h * crop_w * c;
  image_crop_u8_kernel<<<grid_for(total, 256), 256, 0, STREAM>>>(
      src, nimg, hs, ws, c, crop_h, crop_w, reinterpret_cast<uint8_t*>(dst_u8), dst_row_stride, dst_img_stride);
  return check_launch("image_crop_u8");
}

extern "C" int dl_conv_tapsum(const float* y, int nimg, int h, int w, int ldy, int nout, const float* bias,
                              void* out, int out_u8, void* stream_) {
  DL_CHECK_ARG(y && bias && out && nimg > 0 && h > 0 && w > 0, "conv_tapsum: bad args");
  DL_CHECK_ARG(nout >= 1 && nout <= 4 && ldy >= 9 * nout, "conv_tapsum: nout in [1,4], ldy >= 9*nout (got %d, %d)", nout, ldy);
  const long long total = (long long)nimg * h * w;
  if (out_u8)
    conv_tapsum_kernel<true><<<grid_for(total, 256), 256, 0, STREAM>>>(y, nimg, h, w, ldy, nout, bias, out);
  else
    conv_tapsum_kernel<false><<<grid_for(total, 256), 256, 0, STREAM>>>(y, nimg, h, w, ldy, nout, bias, out);
  return check_launch("conv_tapsum");
}

extern "C" int dl_cfg_combine(const float* eps_uncond, const float* eps_text, float guidance_scale,
                              float* out, long long n, void* stream_) {
  DL_CHECK_ARG(eps_uncond && eps_text && out, "cfg_combine: null pointer");
  DL_CHECK_ARG(n % 4 == 0, "cfg_combine: n must be a multiple of 4");
  cfg_combine_kernel<<<grid_for(n / 4, 256), 256, 0, STREAM>>>(
      reinterpret_cast<const float4*>(eps_uncond), reinterpret_cast<const float4*>(eps_text),
      guidance_scale, reinterpret_cast<float4*>(out), n / 4);
  return check_launch("cfg_combine");
}

extern "C" int dl_sampler_step(const float* out_uncond, const float* out_text, float guidance_scale, const float* x,
                               const float* x0_prev, const float* noise, float* x_next, float* x0, long long n,
                               const dl_sampler_coeffs* k, void* stream_) {
  DL_CHECK_ARG(out_uncond && x && x_next && x0 && k, "sampler_step: null pointer");
  DL_CHECK_ARG(n > 0 && n % 4 == 0, "sampler_step: n must be a positive multiple of 4 (got %lld)", n);
  const float* ptrs[] = {out_uncond, out_text, x, x0_prev, noise, x_next, x0};
  for (const float* p : ptrs)
    DL_CHECK_ARG(reinterpret_cast<uintptr_t>(p) % 16 == 0, "sampler_step: operands must be 16-byte aligned");
  DL_CHECK_ARG(x0_prev != nullptr || k->c_1 == 0.f, "sampler_step: c_1 != 0 needs x0_prev");
  DL_CHECK_ARG(noise != nullptr || k->c_n == 0.f, "sampler_step: c_n != 0 needs noise");
  DL_CHECK_ARG(!k->clip_sample || k->clip_sample_range >= 0.f, "sampler_step: clip_sample_range must be >= 0");
  sampler_step_kernel<<<grid_for(n / 4, 256), 256, 0, STREAM>>>(
      reinterpret_cast<const float4*>(out_uncond), reinterpret_cast<const float4*>(out_text), guidance_scale,
      reinterpret_cast<const float4*>(x), reinterpret_cast<const float4*>(x0_prev),
      reinterpret_cast<const float4*>(noise), reinterpret_cast<float4*>(x_next), reinterpret_cast<float4*>(x0),
      n / 4, *k);
  return check_launch("sampler_step");
}

extern "C" int dl_latent_pool8(const float* lat, int nimg, int h, int w, int c, void* out_f16,
                               void* stream_) {
  DL_CHECK_ARG(lat && out_f16 && h > 0 && w > 0 && nimg > 0 && c > 0, "latent_pool8: bad args");
  const int total = nimg * c * 64;
  latent_pool8_kernel<<<(total + 127) / 128, 128, 0, STREAM>>>(lat, nimg, h, w, c,
                                                                reinterpret_cast<__half*>(out_f16));
  return check_launch("latent_pool8");
}
