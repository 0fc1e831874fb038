// Image-to-image entry of the VAE encoder (diffusers LatentConsistencyModelImg2ImgPipeline): the u8 init
// image straight into the im2col operand of conv_in, and the posterior sample + add_noise tail that turns
// the encoder's moments into the first latents of the LCM loop.
#include "common.cuh"
#include "dreamlab_b200.h"

namespace dl {

// cols[p, k] for k = tap*3 + c < 27 (tap = ky*3 + kx of the 3x3 window around pixel p, zero padding outside the
// h x w window), 0 for 27 <= k < 64.  Each value is VaeImageProcessor's 2 * (u8 / 255) - 1 with IEEE division and
// no contraction; the zero padding applies to the normalised image (out-of-window taps are 0.0, not -1).
// One thread per 8 consecutive k of one pixel.
// mask (inpainting, nullable): u8 [nimg, h, w] at its own strides; a pixel with m >= 128 reads as 0.0 before the
// zero padding (StableDiffusionInpaintPipeline's masked_image = image * (binarised mask < 0.5)).
template <typename T>
__global__ void pack_image_im2col_kernel(const uint8_t* __restrict__ img, int nimg, int h, int w,
                                         long long row_stride, long long img_stride, T* __restrict__ out,
                                         const uint8_t* __restrict__ mask, long long mask_row_stride,
                                         long long mask_img_stride) {
  const long long total = (long long)nimg * h * w * 8;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int g = (int)(i & 7);
    const long long p = i >> 3;
    const int x = (int)(p % w);
    const long long r = p / w;
    const int y = (int)(r % h);
    const int n = (int)(r / h);
    float v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int k = g * 8 + j;
      v[j] = 0.f;
      if (k < 27) {
        const int tap = k / 3, c = k % 3;
        const int yi = y + tap / 3 - 1, xi = x + tap % 3 - 1;
        if (yi >= 0 && yi < h && xi >= 0 && xi < w &&
            (mask == nullptr || mask[n * mask_img_stride + yi * mask_row_stride + xi] < 128)) {
          const float u = (float)img[n * img_stride + yi * row_stride + 3LL * xi + c];
          v[j] = __fsub_rn(__fmul_rn(2.f, __fdiv_rn(u, 255.f)), 1.f);
        }
      }
    }
    T* o = out + p * 64 + g * 8;
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

// DiagonalGaussianDistribution.sample + scaling_factor + LCMScheduler.add_noise, one pass.
// moments NHWC [n,h,w,8] (mean | logvar), eps_s / eps_n NCHW [n,4,h,w]; out (and mean_out) NHWC [n,h,w,4].
__global__ void vae_sample_latents_kernel(const float* __restrict__ mom, const float* __restrict__ eps_s,
                                          const float* __restrict__ eps_n, int nimg, int h, int w, float sf,
                                          float sqrt_a, float sqrt_b, float* __restrict__ out,
                                          float* __restrict__ mean_out) {
  const long long hw = (long long)h * w;
  const long long total = nimg * hw * 4;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(i & 3);
    const long long p = i >> 2;                       // n * hw + pixel
    const long long n = p / hw, q = p % hw;
    const float mean = mom[p * 8 + c];
    const float lv = fminf(fmaxf(mom[p * 8 + 4 + c], -30.f), 20.f);
    const float sd = expf(__fmul_rn(0.5f, lv));
    const long long e = (n * 4 + c) * hw + q;
    const float x0 = __fmul_rn(sf, __fadd_rn(mean, __fmul_rn(sd, eps_s[e])));
    out[i] = __fadd_rn(__fmul_rn(sqrt_a, x0), __fmul_rn(sqrt_b, eps_n[e]));
    if (mean_out) mean_out[i] = mean;
  }
}

static inline unsigned i2i_grid(long long total, int threads) {
  long long b = (total + threads - 1) / threads;
  const long long cap = (long long)num_sms() * 32;
  if (b > cap) b = cap;
  if (b < 1) b = 1;
  return (unsigned)b;
}

}  // namespace dl

using namespace dl;
#define STREAM reinterpret_cast<cudaStream_t>(stream_)

extern "C" int dl_pack_image_im2col(const void* img_u8, int nimg, int h, int w, long long row_stride,
                                    long long img_stride, void* out, void* stream_) {
  DL_CHECK_ARG(img_u8 && out && nimg > 0 && h > 0 && w > 0 && row_stride >= 3LL * w &&
               (nimg == 1 || img_stride >= row_stride * h), "pack_image_im2col: bad args");
  const long long total = (long long)nimg * h * w * 8;
  pack_image_im2col_kernel<__nv_bfloat16><<<i2i_grid(total, 256), 256, 0, STREAM>>>(
      reinterpret_cast<const uint8_t*>(img_u8), nimg, h, w, row_stride, img_stride,
      reinterpret_cast<__nv_bfloat16*>(out), nullptr, 0, 0);
  return check_launch("pack_image_im2col");
}

extern "C" int dl_pack_image_im2col_f32(const void* img_u8, int nimg, int h, int w, long long row_stride,
                                        long long img_stride, float* out, void* stream_) {
  DL_CHECK_ARG(img_u8 && out && nimg > 0 && h > 0 && w > 0 && row_stride >= 3LL * w &&
               (nimg == 1 || img_stride >= row_stride * h), "pack_image_im2col_f32: bad args");
  const long long total = (long long)nimg * h * w * 8;
  pack_image_im2col_kernel<float><<<i2i_grid(total, 256), 256, 0, STREAM>>>(
      reinterpret_cast<const uint8_t*>(img_u8), nimg, h, w, row_stride, img_stride, out, nullptr, 0, 0);
  return check_launch("pack_image_im2col_f32");
}

extern "C" int dl_pack_image_im2col_masked(const void* img_u8, const void* mask_u8, int nimg, int h, int w,
                                           long long row_stride, long long img_stride, long long mask_row_stride,
                                           long long mask_img_stride, void* out, void* stream_) {
  DL_CHECK_ARG(img_u8 && mask_u8 && out && nimg > 0 && h > 0 && w > 0 && row_stride >= 3LL * w &&
               (nimg == 1 || img_stride >= row_stride * h) && mask_row_stride >= w &&
               (nimg == 1 || mask_img_stride >= mask_row_stride * h), "pack_image_im2col_masked: bad args");
  const long long total = (long long)nimg * h * w * 8;
  pack_image_im2col_kernel<__nv_bfloat16><<<i2i_grid(total, 256), 256, 0, STREAM>>>(
      reinterpret_cast<const uint8_t*>(img_u8), nimg, h, w, row_stride, img_stride,
      reinterpret_cast<__nv_bfloat16*>(out), reinterpret_cast<const uint8_t*>(mask_u8), mask_row_stride,
      mask_img_stride);
  return check_launch("pack_image_im2col_masked");
}

extern "C" int dl_pack_image_im2col_masked_f32(const void* img_u8, const void* mask_u8, int nimg, int h, int w,
                                               long long row_stride, long long img_stride, long long mask_row_stride,
                                               long long mask_img_stride, float* out, void* stream_) {
  DL_CHECK_ARG(img_u8 && mask_u8 && out && nimg > 0 && h > 0 && w > 0 && row_stride >= 3LL * w &&
               (nimg == 1 || img_stride >= row_stride * h) && mask_row_stride >= w &&
               (nimg == 1 || mask_img_stride >= mask_row_stride * h), "pack_image_im2col_masked_f32: bad args");
  const long long total = (long long)nimg * h * w * 8;
  pack_image_im2col_kernel<float><<<i2i_grid(total, 256), 256, 0, STREAM>>>(
      reinterpret_cast<const uint8_t*>(img_u8), nimg, h, w, row_stride, img_stride, out,
      reinterpret_cast<const uint8_t*>(mask_u8), mask_row_stride, mask_img_stride);
  return check_launch("pack_image_im2col_masked_f32");
}

extern "C" int dl_vae_sample_latents(const float* moments, const float* eps_s, const float* eps_n, int nimg, int h,
                                     int w, float scaling_factor, float sqrt_alpha, float sqrt_one_minus_alpha,
                                     float* out, float* mean_out, void* stream_) {
  DL_CHECK_ARG(moments && eps_s && eps_n && out && nimg > 0 && h > 0 && w > 0, "vae_sample_latents: bad args");
  const long long total = (long long)nimg * h * w * 4;
  vae_sample_latents_kernel<<<i2i_grid(total, 256), 256, 0, STREAM>>>(
      moments, eps_s, eps_n, nimg, h, w, scaling_factor, sqrt_alpha, sqrt_one_minus_alpha, out, mean_out);
  return check_launch("vae_sample_latents");
}
