// b200seg — GPU input pipeline (SURVEY.md §8f N4): the reference's segmentation training transform
//   A.Resize(256,256) -> A.ShiftScaleRotate(0.05, 0.05, 15deg, p=0.7) -> A.HorizontalFlip(0.5)
//   -> A.RandomBrightnessContrast(0.1, 0.1, p=0.5) -> A.Normalize(ImageNet) -> ToTensorV2      (utils/trainer.py:88-101)
// and the mask's `/ 255` (utils/dataset.py:124-126), as ONE kernel per batch: raw uint8 HWC images + uint8 masks in,
// normalised fp32 NCHW image + fp32 {0..1} mask out (the layout the model's stem kernels read).  At ~2 k images/s per
// GPU the reference's 4-worker PIL / Albumentations loader (a few hundred images/s) cannot feed the training step.
//
// The uint8 rounding points of the CPU pipeline are reproduced: the resize result is rounded to uint8 (cv2.resize,
// INTER_LINEAR, half-pixel centres), the affine warp samples THAT image with coordinates quantised to 1/32 pixel and
// BORDER_REFLECT_101 (cv2.warpAffine as Albumentations calls it; INTER_NEAREST for the mask), the flip mirrors the warped
// image, brightness / contrast go through the uint8 look-up table of Albumentations (truncating cast), and only then
// the image is normalised in fp32.  Random parameters are drawn on the host (per-sample inverse affine matrix, flip,
// alpha, beta): the kernel is deterministic.
#include "common.cuh"

namespace b2 {

struct AugSample {      // per image, mirrors b2_aug_params
  float m[6];           // INVERSE affine: (xs, ys) = (m0*x + m1*y + m2, m3*x + m4*y + m5) in the resized S x S image
  float alpha, beta;    // v' = clip(alpha * v + beta * 255), uint8 LUT
  int flip, warp, adjust, border;   // border: 0 = cv2.BORDER_CONSTANT (fill 0; Albumentations 2.x default), 1 = REFLECT_101
};

__device__ __forceinline__ int reflect101(int i, int n) {
  if (n == 1) return 0;
  while (i < 0 || i >= n) i = i < 0 ? -i : 2 * n - 2 - i;
  return i;
}

// value of channel c of the RESIZED (S x S) image at integer pixel (yy, xx): bilinear from the source, rounded to uint8
__device__ __forceinline__ float resized_u8(const uint8_t* __restrict__ img, int hs, int ws, int ch, int c, int yy, int xx,
                                            float sy, float sx) {
  float fy = (yy + 0.5f) * sy - 0.5f, fx = (xx + 0.5f) * sx - 0.5f;
  int y0 = (int)floorf(fy), x0 = (int)floorf(fx);
  float wy = fy - y0, wx = fx - x0;
  if (y0 < 0) { y0 = 0; wy = 0.f; }
  if (x0 < 0) { x0 = 0; wx = 0.f; }
  int y1 = y0 + 1, x1 = x0 + 1;
  if (y1 >= hs) { y1 = hs - 1; if (y0 >= hs - 1) { y0 = hs - 1; wy = 0.f; } }
  if (x1 >= ws) { x1 = ws - 1; if (x0 >= ws - 1) { x0 = ws - 1; wx = 0.f; } }
  const float v00 = img[((long long)y0 * ws + x0) * ch + c], v01 = img[((long long)y0 * ws + x1) * ch + c];
  const float v10 = img[((long long)y1 * ws + x0) * ch + c], v11 = img[((long long)y1 * ws + x1) * ch + c];
  const float v = (v00 * (1.f - wx) + v01 * wx) * (1.f - wy) + (v10 * (1.f - wx) + v11 * wx) * wy;
  return floorf(v + 0.5f);
}

__device__ __forceinline__ float resized_mask(const uint8_t* __restrict__ msk, int hs, int ws, int yy, int xx, float sy,
                                              float sx, int nearest) {
  if (nearest) {          // cv2.resize INTER_NEAREST: src = floor(dst * scale)
    int y = (int)floorf(yy * sy), x = (int)floorf(xx * sx);
    y = y < hs ? y : hs - 1;
    x = x < ws ? x : ws - 1;
    return (float)msk[(long long)y * ws + x];
  }
  return resized_u8(msk, hs, ws, 1, 0, yy, xx, sy, sx);
}

// kLabels: the mask is a class-index map (nearest resize, written as uint8 to `t`); otherwise {0, 255} -> fp32 {0, 1}
template <bool kLabels>
__global__ void __launch_bounds__(256) seg_augment_kernel(const uint8_t* __restrict__ img, const uint8_t* __restrict__ msk,
                                                          int n, int hs, int ws, int S, const AugSample* __restrict__ prm,
                                                          float3 mean, float3 inv_std, int mask_nearest_resize,
                                                          float* __restrict__ x, void* __restrict__ t) {
  const long long total = (long long)n * S * S;
  const float sy = (float)hs / S, sx = (float)ws / S;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int xo = (int)(i % S);
    const int yo = (int)((i / S) % S);
    const int b = (int)(i / ((long long)S * S));
    const AugSample a = prm[b];
    const uint8_t* im = img + (long long)b * hs * ws * 3;
    const uint8_t* mk = msk + (long long)b * hs * ws;
    const int xw = a.flip ? S - 1 - xo : xo;           // HorizontalFlip acts on the warped image
    float rgb[3], mv;
    if (a.warp) {
      // cv2.warpAffine: source coordinates rounded to 1/32 pixel, bilinear, BORDER_REFLECT_101
      const float fx = a.m[0] * xw + a.m[1] * yo + a.m[2], fy = a.m[3] * xw + a.m[4] * yo + a.m[5];
      const int X = (int)lrintf(fx * 32.f), Y = (int)lrintf(fy * 32.f);
      const int x0 = X >> 5, y0 = Y >> 5;
      const float wx = (X & 31) * (1.f / 32.f), wy = (Y & 31) * (1.f / 32.f);
      const bool refl = a.border != 0;
      const int xa = refl ? reflect101(x0, S) : x0, xb = refl ? reflect101(x0 + 1, S) : x0 + 1;
      const int ya = refl ? reflect101(y0, S) : y0, yb = refl ? reflect101(y0 + 1, S) : y0 + 1;
      const bool ixa = xa >= 0 && xa < S, ixb = xb >= 0 && xb < S, iya = ya >= 0 && ya < S, iyb = yb >= 0 && yb < S;
#pragma unroll
      for (int c = 0; c < 3; ++c) {      // taps outside the image are the constant border (0)
        const float v00 = (iya && ixa) ? resized_u8(im, hs, ws, 3, c, ya, xa, sy, sx) : 0.f;
        const float v01 = (iya && ixb) ? resized_u8(im, hs, ws, 3, c, ya, xb, sy, sx) : 0.f;
        const float v10 = (iyb && ixa) ? resized_u8(im, hs, ws, 3, c, yb, xa, sy, sx) : 0.f;
        const float v11 = (iyb && ixb) ? resized_u8(im, hs, ws, 3, c, yb, xb, sy, sx) : 0.f;
        rgb[c] = floorf((v00 * (1.f - wx) + v01 * wx) * (1.f - wy) + (v10 * (1.f - wx) + v11 * wx) * wy + 0.5f);
      }
      // mask: INTER_NEAREST in the warp (cv2 rounds the 1/32-quantised coordinate to the nearest pixel)
      int xn = (X + 16) >> 5, yn = (Y + 16) >> 5;
      if (refl) { xn = reflect101(xn, S); yn = reflect101(yn, S); }
      mv = (xn >= 0 && xn < S && yn >= 0 && yn < S) ? resized_mask(mk, hs, ws, yn, xn, sy, sx, mask_nearest_resize) : 0.f;
    } else {
#pragma unroll
      for (int c = 0; c < 3; ++c) rgb[c] = resized_u8(im, hs, ws, 3, c, yo, xw, sy, sx);
      mv = resized_mask(mk, hs, ws, yo, xw, sy, sx, mask_nearest_resize);
    }
    if (a.adjust) {
#pragma unroll
      for (int c = 0; c < 3; ++c) rgb[c] = floorf(fminf(fmaxf(rgb[c] * a.alpha + a.beta * 255.f, 0.f), 255.f));
    }
    const long long plane = (long long)S * S, o = (long long)yo * S + xo;
    x[((long long)b * 3 + 0) * plane + o] = (rgb[0] * (1.f / 255.f) - mean.x) * inv_std.x;
    x[((long long)b * 3 + 1) * plane + o] = (rgb[1] * (1.f / 255.f) - mean.y) * inv_std.y;
    x[((long long)b * 3 + 2) * plane + o] = (rgb[2] * (1.f / 255.f) - mean.z) * inv_std.z;
    if constexpr (kLabels) static_cast<uint8_t*>(t)[(long long)b * plane + o] = (uint8_t)mv;
    else static_cast<float*>(t)[(long long)b * plane + o] = mv * (1.f / 255.f);
  }
}

static int seg_augment(bool labels, const uint8_t* img, const uint8_t* mask, int32_t n, int32_t hs, int32_t ws,
                       int32_t size, const b2_aug_params* params, const float* mean3, const float* std3,
                       int32_t mask_nearest_resize, float* x, void* t, b2_stream_t stream) {
  static_assert(sizeof(AugSample) == sizeof(b2_aug_params), "AugSample must mirror b2_aug_params");
  int rc = b2_arch_check();
  if (rc) return rc;
  B2_REQUIRE(n > 0 && hs > 0 && ws > 0 && size > 0 && mean3 != nullptr && std3 != nullptr, B2_ERR_SHAPE,
             "bad augmentation request");
  const long long total = (long long)n * size * size;
  long long grid = (total + 255) / 256;
  const long long cap = (long long)num_sms() * 16;
  if (grid > cap) grid = cap;
  const float3 mean = make_float3(mean3[0], mean3[1], mean3[2]);
  const float3 inv_std = make_float3(1.f / std3[0], 1.f / std3[1], 1.f / std3[2]);
  const AugSample* prm = reinterpret_cast<const AugSample*>(params);
  if (labels)
    seg_augment_kernel<true><<<(unsigned)grid, 256, 0, (cudaStream_t)stream>>>(img, mask, n, hs, ws, size, prm, mean,
                                                                              inv_std, mask_nearest_resize, x, t);
  else
    seg_augment_kernel<false><<<(unsigned)grid, 256, 0, (cudaStream_t)stream>>>(img, mask, n, hs, ws, size, prm, mean,
                                                                               inv_std, mask_nearest_resize, x, t);
  B2_LAUNCH_CHECK();
  return B2_OK;
}

}  // namespace b2

using namespace b2;

extern "C" int b2_seg_augment(const uint8_t* img, const uint8_t* mask, int32_t n, int32_t hs, int32_t ws, int32_t size,
                              const b2_aug_params* params, const float* mean3, const float* std3,
                              int32_t mask_nearest_resize, float* x, float* t, b2_stream_t stream) {
  return seg_augment(false, img, mask, n, hs, ws, size, params, mean3, std3, mask_nearest_resize, x, t, stream);
}

extern "C" int b2_seg_augment_labels(const uint8_t* img, const uint8_t* mask, int32_t n, int32_t hs, int32_t ws,
                                     int32_t size, const b2_aug_params* params, const float* mean3, const float* std3,
                                     float* x, uint8_t* labels, b2_stream_t stream) {
  return seg_augment(true, img, mask, n, hs, ws, size, params, mean3, std3, 1, x, labels, stream);
}
