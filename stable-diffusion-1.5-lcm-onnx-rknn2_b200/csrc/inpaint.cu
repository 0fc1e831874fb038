// Inpainting side kernels (diffusers StableDiffusionInpaintPipeline with LCMScheduler): the latent mask, the
// 9-channel conv_in operand [latents | mask | masked_image_latents], and LCMScheduler.step fused with the 4-channel
// UNet's blend towards the noised image latents.  The masked encoder input is `dl_pack_image_im2col_masked`
// (img2img.cu), the posterior samples are `dl_vae_sample_latents`.
#include "common.cuh"
#include "dreamlab_b200.h"

namespace dl {

// mask_processor (grayscale, / 255, binarise at 0.5) + F.interpolate(size=(H/8, W/8), mode="nearest"):
// out[n, i, j] = mask[n, 8i, 8j] >= 128 ? 1 : 0.
__global__ void inpaint_latent_mask_kernel(const uint8_t* __restrict__ mask, int nimg, int h, int w,
                                           float* __restrict__ out) {
  const long long total = (long long)nimg * h * w;
  const long long W = 8LL * w, HW = 64LL * h * w;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int x = (int)(i % w);
    const long long r = i / w;
    const int y = (int)(r % h);
    const long long n = r / h;
    out[i] = mask[n * HW + 8LL * y * W + 8LL * x] >= 128 ? 1.f : 0.f;
  }
}

// out[(r*nimg + n), y, x, c] for r < repeat: c < 4 latents, c == 4 mask, 5 <= c < 9 masked latents, 0 up to 64.
// latents / masked fp32 NHWC [nimg,h,w,4], mask fp32 [nimg,h,w].  One thread per 8 consecutive channels.
template <typename T>
__global__ void pack_latent_inpaint_kernel(const float* __restrict__ lat, const float* __restrict__ mask,
                                           const float* __restrict__ masked, long long npix, int repeat,
                                           T* __restrict__ out) {
  const long long total = npix * repeat * 8;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int g = (int)(i & 7);
    const long long q = i >> 3;                 // output pixel
    const long long p = q % npix;               // source pixel (every repeat packs the same latents)
    float v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int c = g * 8 + j;
      v[j] = c < 4 ? lat[p * 4 + c] : c == 4 ? mask[p] : c < 9 ? masked[p * 4 + c - 5] : 0.f;
    }
    T* o = out + q * 64 + g * 8;
    if constexpr (sizeof(T) == 4) {
      reinterpret_cast<float4*>(o)[0] = make_float4(v[0], v[1], v[2], v[3]);
      reinterpret_cast<float4*>(o)[1] = make_float4(v[4], v[5], v[6], v[7]);
    } else {
      uint4 u;
      u.x = pack_bf16x2(v[0], v[1]);
      u.y = pack_bf16x2(v[2], v[3]);
      u.z = pack_bf16x2(v[4], v[5]);
      u.w = pack_bf16x2(v[6], v[7]);
      *reinterpret_cast<uint4*>(o) = u;
    }
  }
}

// LCMScheduler.step (same op order as lcm_step_kernel), then the 4-channel UNet's blend:
//   proper = last ? image_latents : sqrt_a * image_latents + sqrt_b * noise0        (add_noise at timesteps[i+1])
//   x_next = (1 - m) * proper + m * prev_sample
// fp32 NHWC [.., 4] tensors as float4 (one pixel each), mask fp32 one value per pixel.
__global__ void lcm_step_inpaint_kernel(const float4* __restrict__ eps, const float4* __restrict__ x,
                                        const float4* __restrict__ noise, const float4* __restrict__ img,
                                        const float4* __restrict__ noise0, const float* __restrict__ mask,
                                        float4* __restrict__ x_next, float4* __restrict__ denoised, long long n4,
                                        dl_lcm_coeffs k, float sqrt_a, float sqrt_b, int last) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4;
       i += (long long)gridDim.x * blockDim.x) {
    const float4 e = eps[i], xv = x[i], iv = img[i];
    const float ev[4] = {e.x, e.y, e.z, e.w};
    const float xx[4] = {xv.x, xv.y, xv.z, xv.w};
    const float im[4] = {iv.x, iv.y, iv.z, iv.w};
    float zz[4] = {0.f, 0.f, 0.f, 0.f}, z0[4] = {0.f, 0.f, 0.f, 0.f};
    if (noise != nullptr) {
      const float4 z = noise[i];
      zz[0] = z.x; zz[1] = z.y; zz[2] = z.z; zz[3] = z.w;
    }
    if (!last) {
      const float4 z = noise0[i];
      z0[0] = z.x; z0[1] = z.y; z0[2] = z.z; z0[3] = z.w;
    }
    const float m = mask[i];
    const float m1 = __fsub_rn(1.f, m);
    float d[4], o[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float x0 = __fdiv_rn(__fsub_rn(xx[j], __fmul_rn(k.sqrt_beta_t, ev[j])), k.sqrt_alpha_t);
      d[j] = __fadd_rn(__fmul_rn(k.c_out, x0), __fmul_rn(k.c_skip, xx[j]));
      const float prev = (noise != nullptr)
                             ? __fadd_rn(__fmul_rn(k.sqrt_alpha_prev, d[j]), __fmul_rn(k.sqrt_beta_prev, zz[j]))
                             : d[j];
      const float proper = last ? im[j] : __fadd_rn(__fmul_rn(sqrt_a, im[j]), __fmul_rn(sqrt_b, z0[j]));
      o[j] = __fadd_rn(__fmul_rn(m1, proper), __fmul_rn(m, prev));
    }
    denoised[i] = make_float4(d[0], d[1], d[2], d[3]);
    x_next[i] = make_float4(o[0], o[1], o[2], o[3]);
  }
}

static inline unsigned inp_grid(long long total, int threads) {
  long long b = (total + threads - 1) / threads;
  const long long cap = (long long)num_sms() * 32;
  if (b > cap) b = cap;
  if (b < 1) b = 1;
  return (unsigned)b;
}

}  // namespace dl

using namespace dl;
#define STREAM reinterpret_cast<cudaStream_t>(stream_)

extern "C" int dl_inpaint_latent_mask(const void* mask_u8, int nimg, int h, int w, float* out, void* stream_) {
  DL_CHECK_ARG(mask_u8 && out && nimg > 0 && h > 0 && w > 0, "inpaint_latent_mask: bad args");
  const long long total = (long long)nimg * h * w;
  inpaint_latent_mask_kernel<<<inp_grid(total, 256), 256, 0, STREAM>>>(reinterpret_cast<const uint8_t*>(mask_u8),
                                                                      nimg, h, w, out);
  return check_launch("inpaint_latent_mask");
}

extern "C" int dl_pack_latent_inpaint(const float* latents, const float* mask, const float* masked, long long npix,
                                      int repeat, void* out, void* stream_) {
  DL_CHECK_ARG(latents && mask && masked && out && npix > 0 && repeat > 0, "pack_latent_inpaint: bad args");
  const long long total = npix * repeat * 8;
  pack_latent_inpaint_kernel<__nv_bfloat16><<<inp_grid(total, 256), 256, 0, STREAM>>>(
      latents, mask, masked, npix, repeat, reinterpret_cast<__nv_bfloat16*>(out));
  return check_launch("pack_latent_inpaint");
}

extern "C" int dl_pack_latent_inpaint_f32(const float* latents, const float* mask, const float* masked,
                                          long long npix, int repeat, float* out, void* stream_) {
  DL_CHECK_ARG(latents && mask && masked && out && npix > 0 && repeat > 0, "pack_latent_inpaint_f32: bad args");
  const long long total = npix * repeat * 8;
  pack_latent_inpaint_kernel<float><<<inp_grid(total, 256), 256, 0, STREAM>>>(latents, mask, masked, npix, repeat,
                                                                             out);
  return check_launch("pack_latent_inpaint_f32");
}

extern "C" int dl_lcm_step_inpaint(const float* eps, const float* x, const float* noise, const float* image_latents,
                                   const float* noise0, const float* mask, float* x_next, float* denoised,
                                   long long npix, const dl_lcm_coeffs* k, float sqrt_alpha, float sqrt_one_minus_alpha,
                                   int last, void* stream_) {
  DL_CHECK_ARG(eps && x && image_latents && mask && x_next && denoised && k && npix > 0 && (last || noise0),
               "lcm_step_inpaint: bad args");
  lcm_step_inpaint_kernel<<<inp_grid(npix, 256), 256, 0, STREAM>>>(
      reinterpret_cast<const float4*>(eps), reinterpret_cast<const float4*>(x),
      reinterpret_cast<const float4*>(noise), reinterpret_cast<const float4*>(image_latents),
      reinterpret_cast<const float4*>(noise0), mask, reinterpret_cast<float4*>(x_next),
      reinterpret_cast<float4*>(denoised), npix, *k, sqrt_alpha, sqrt_one_minus_alpha, last);
  return check_launch("lcm_step_inpaint");
}
