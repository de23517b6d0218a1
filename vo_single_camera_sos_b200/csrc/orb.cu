// ORB description of given keypoints on the panoramas (SURVEY §8f row N3, description half).
//
// replaces: descriptor.compute(image = pano_img, keypoints = ...) with descriptor = cv2.ORB_create(nfeatures)
//           in OmniCamModel.detect_sparse_features_on_panorama (camera_models.py:1680-1683, 1766) and
//           cv2.cvtColor(pano_img, COLOR_BGR2GRAY) (camera_models.py:1711).
//
// What cv2.ORB.compute does with user-supplied keypoints of octave 0 was identified from its behaviour and is pinned bit
// for bit by scripts/derive_orb_pattern.py (409 600 descriptor bits, zero differences):
//   * keypoints closer than 31 px to the image border are dropped (KeyPointsFilter::runByImageBorder, edgeThreshold);
//   * the image is blurred by the separable 7-tap Gaussian of sigma 2 (BORDER_REFLECT_101) — evaluated exactly and
//     rounded once, NOT cv2.GaussianBlur's fixed-point path;
//   * orientation is NOT recomputed: the keypoint's own angle is used (-1 degree for cv2.KeyPoint_convert points, i.e.
//     the reference's default GFT detector);
//   * bit k = B[c + round(R p0_k)] < B[c + round(R p1_k)] with c = cvRound(keypoint), R the rotation by the angle in float32
//     arithmetic without contraction, round = cvRound (half to even), 8 bits per byte, first test in the LSB.
#include <math_constants.h>

#include "sos_common.cuh"

namespace {

__constant__ int8_t c_orb_pattern[256 * 4] = {
#include "orb_pattern.inc"
};

constexpr int ORB_EDGE = 31;

// cv::cvtColor(BGR2GRAY) for 8-bit images in OpenCV 4.x: fixed point with 15 fractional bits (B 3735, G 19235, R 9798)
__device__ __forceinline__ uint32_t gray_of(uint32_t b, uint32_t g, uint32_t r) {
  return (b * 3735u + g * 19235u + r * 9798u + 16384u) >> 15;
}

// four pixels per thread: three aligned 32-bit loads, one 32-bit store (the scalar form issued three strided byte loads per
// pixel: 0.18 ms for 32 C2 panoramas)
__global__ void bgr2gray_kernel(const uint8_t* __restrict__ bgr, size_t n, uint8_t* __restrict__ gray, int vec_ok) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t p = 4 * i;
  if (p >= n) return;
  if (vec_ok && p + 4 <= n) {
    const uint32_t* w = (const uint32_t*)(bgr + 3 * p);
    const uint32_t w0 = __ldg(w), w1 = __ldg(w + 1), w2 = __ldg(w + 2);
    const uint32_t g0 = gray_of(w0 & 255u, (w0 >> 8) & 255u, (w0 >> 16) & 255u);
    const uint32_t g1 = gray_of(w0 >> 24, w1 & 255u, (w1 >> 8) & 255u);
    const uint32_t g2 = gray_of((w1 >> 16) & 255u, w1 >> 24, w2 & 255u);
    const uint32_t g3 = gray_of((w2 >> 8) & 255u, (w2 >> 16) & 255u, w2 >> 24);
    *(uint32_t*)(gray + p) = g0 | (g1 << 8) | (g2 << 16) | (g3 << 24);
  } else {
    for (size_t q = p; q < n && q < p + 4; ++q) gray[q] = (uint8_t)gray_of(bgr[3 * q], bgr[3 * q + 1], bgr[3 * q + 2]);
  }
}

__device__ __forceinline__ int reflect101(int p, int n) {
  if (n == 1) return 0;
  while (p < 0 || p >= n) p = p < 0 ? -p : 2 * n - 2 - p;
  return p;
}

struct Gauss7 {
  double k[7];
};

constexpr int BL_ROWS = 32, BL_R = 3;

// out = round_half_even(G * in), exact separable convolution in float64 (horizontal pass, then vertical, taps in order).
// One thread per column walks down a strip of BL_ROWS rows with the horizontal sums of the last seven rows in registers; the
// next row's seven taps are loaded one iteration ahead.  (First version: 64 x 16 tiles with the horizontal sums staged as
// doubles in shared memory, 0.43 ms for 32 C2 panoramas.)
__global__ void __launch_bounds__(128) orb_blur_kernel(const uint8_t* __restrict__ in, int H, int W, Gauss7 g,
                                                       uint8_t* __restrict__ out) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  if (x >= W) return;
  const int y0 = blockIdx.y * BL_ROWS, y1 = min(H, y0 + BL_ROWS);
  const uint8_t* src = in + (size_t)blockIdx.z * H * W;
  uint8_t* dst = out + (size_t)blockIdx.z * H * W;
  int cx[7];
#pragma unroll
  for (int t = 0; t < 7; ++t) cx[t] = reflect101(x + t - BL_R, W);
  uint8_t raw[7];
  auto fetch = [&](int row) {
    const uint8_t* r = src + (size_t)reflect101(row, H) * W;
#pragma unroll
    for (int t = 0; t < 7; ++t) raw[t] = __ldg(r + cx[t]);
  };
  auto hsum = [&]() {
    double s = 0.0;
#pragma unroll
    for (int t = 0; t < 7; ++t) s += g.k[t] * (double)raw[t];
    return s;
  };
  double h[7];
#pragma unroll
  for (int t = 0; t < 6; ++t) {
    fetch(y0 - BL_R + t);
    h[t] = hsum();
  }
  fetch(y0 + BL_R);
  for (int y = y0; y < y1; ++y) {
    h[6] = hsum();                                       // row y + 3
    fetch(y + BL_R + 1);
    double s = 0.0;
#pragma unroll
    for (int t = 0; t < 7; ++t) s += g.k[t] * h[t];
    const int v = __double2int_rn(s);
    dst[(size_t)y * W + x] = (uint8_t)min(255, max(0, v));
#pragma unroll
    for (int t = 0; t < 6; ++t) h[t] = h[t + 1];
  }
}

// one warp per keypoint, one descriptor byte per lane
__global__ void __launch_bounds__(256)
orb_describe_kernel(const uint8_t* __restrict__ blurred, int H, int W, const float2* __restrict__ kp,
                    const float* __restrict__ angle_deg, const int32_t* __restrict__ img_idx, int n,
                    uint32_t* __restrict__ desc, uint8_t* __restrict__ keep) {
  // without per-keypoint angles (cv2.KeyPoint_convert: -1 degree for all) the rotated test offsets are the same for every
  // keypoint: computed once per block
  __shared__ int s_off[512];
  if (!angle_deg) {
    const float ang0 = __fmul_rn(-1.0f, (float)(CUDART_PI / 180.0f));
    const float a0 = (float)cos((double)ang0), b0 = (float)sin((double)ang0);
    for (int q = threadIdx.x; q < 512; q += blockDim.x) {
      const float px = (float)c_orb_pattern[2 * q], py = (float)c_orb_pattern[2 * q + 1];
      const int ix = __float2int_rn(__fsub_rn(__fmul_rn(px, a0), __fmul_rn(py, b0)));
      const int iy = __float2int_rn(__fadd_rn(__fmul_rn(px, b0), __fmul_rn(py, a0)));
      s_off[q] = iy * W + ix;
    }
    __syncthreads();
  }
  const int i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (i >= n) return;
  const float2 p = kp[i];
  // KeyPointsFilter::runByImageBorder: Rect(31, 31, W - 62, H - 62).contains(Point(pt)) — the Point2f is first converted to an
  // integer point with cvRound (probed: x = 30.5 is dropped, 30.51 kept, 388.5 kept and 388.99 dropped at W = 420)
  const int rx = __float2int_rn(p.x), ry = __float2int_rn(p.y);
  const bool inside = rx >= ORB_EDGE && rx < W - ORB_EDGE && ry >= ORB_EDGE && ry < H - ORB_EDGE;
  if (lane == 0 && keep) keep[i] = inside ? 1 : 0;
  uint32_t byte = 0;
  if (inside) {
    const uint8_t* img = blurred + (size_t)(img_idx ? img_idx[i] : 0) * H * W;
    const int cx = __float2int_rn(p.x), cy = __float2int_rn(p.y);
    float ang = angle_deg ? angle_deg[i] : -1.0f;
    ang = __fmul_rn(ang, (float)(CUDART_PI / 180.0f));
    const float a = (float)cos((double)ang), b = (float)sin((double)ang);
    const uint8_t* center = img + (size_t)cy * W + cx;
    if (!angle_deg) {
#pragma unroll
      for (int t = 0; t < 8; ++t) {
        const int q = (lane * 8 + t) * 2;
        const uint32_t v0 = center[s_off[q]], v1 = center[s_off[q + 1]];
        byte |= (v0 < v1 ? 1u : 0u) << t;
      }
    } else
#pragma unroll
    for (int t = 0; t < 8; ++t) {
      const int k = (lane * 8 + t) * 4;
      const float px0 = (float)c_orb_pattern[k], py0 = (float)c_orb_pattern[k + 1];
      const float px1 = (float)c_orb_pattern[k + 2], py1 = (float)c_orb_pattern[k + 3];
      const int ix0 = __float2int_rn(__fsub_rn(__fmul_rn(px0, a), __fmul_rn(py0, b)));
      const int iy0 = __float2int_rn(__fadd_rn(__fmul_rn(px0, b), __fmul_rn(py0, a)));
      const int ix1 = __float2int_rn(__fsub_rn(__fmul_rn(px1, a), __fmul_rn(py1, b)));
      const int iy1 = __float2int_rn(__fadd_rn(__fmul_rn(px1, b), __fmul_rn(py1, a)));
      const uint32_t v0 = center[iy0 * W + ix0], v1 = center[iy1 * W + ix1];
      byte |= (v0 < v1 ? 1u : 0u) << t;
    }
  }
  // four consecutive lanes -> one little-endian word
  uint32_t word = byte << (8 * (lane & 3));
  word |= __shfl_xor_sync(0xFFFFFFFFu, word, 1);
  word |= __shfl_xor_sync(0xFFFFFFFFu, word, 2);
  if ((lane & 3) == 0) desc[(size_t)i * 8 + (lane >> 2)] = word;
}

Gauss7 gauss_7_sigma2() {
  Gauss7 g;
  double sum = 0.0;
  for (int t = 0; t < 7; ++t) {
    const double x = (double)(t - 3);
    g.k[t] = exp(-(x * x) / (2.0 * 2.0 * 2.0));
    sum += g.k[t];
  }
  for (int t = 0; t < 7; ++t) g.k[t] /= sum;
  return g;
}

}  // namespace

extern "C" int sos_bgr_to_gray(sos_ctx* ctx, const uint8_t* bgr, size_t n_pixels, uint8_t* gray) {
  SOS_CHECK_ARG(ctx, "ctx is NULL");
  if (n_pixels == 0) return SOS_OK;
  SOS_CHECK_ARG(bgr && gray, "NULL array");
  SOS_CHECK_ARG(n_pixels / 256 < (1ull << 31), "image too large");
  SOS_CUDA(cudaSetDevice(ctx->device));
  const int vec_ok = ((uintptr_t)bgr % 4 == 0) && ((uintptr_t)gray % 4 == 0);
  const size_t n_thr = (n_pixels + 3) / 4;
  bgr2gray_kernel<<<(unsigned)((n_thr + 255) / 256), 256, 0, ctx->stream>>>(bgr, n_pixels, gray, vec_ok);
  SOS_LAUNCHED_AS(ctx, "bgr2gray_kernel");
  return SOS_OK;
}

extern "C" int sos_orb_blur(sos_ctx* ctx, const uint8_t* gray, int n_images, int height, int width, uint8_t* blurred) {
  SOS_CHECK_ARG(ctx, "ctx is NULL");
  SOS_CHECK_ARG(n_images >= 0 && height >= 0 && width >= 0, "negative size");
  if (n_images == 0 || height == 0 || width == 0) return SOS_OK;
  SOS_CHECK_ARG(gray && blurred && gray != blurred, "NULL array or in-place call");
  SOS_CHECK_ARG(n_images <= 65535 && sos_div_up(height, BL_ROWS) <= 65535, "too many images / rows");
  SOS_CUDA(cudaSetDevice(ctx->device));
  dim3 grid(sos_div_up(width, 128), sos_div_up(height, BL_ROWS), n_images);
  orb_blur_kernel<<<grid, 128, 0, ctx->stream>>>(gray, height, width, gauss_7_sigma2(), blurred);
  SOS_LAUNCHED_AS(ctx, "orb_blur_kernel");
  return SOS_OK;
}

extern "C" int sos_orb_describe(sos_ctx* ctx, const uint8_t* gray, int n_images, int height, int width, const float* kp_xy,
                                const float* kp_angle_deg, const int32_t* kp_image, int n, uint32_t* desc, uint8_t* keep) {
  SOS_CHECK_ARG(ctx, "ctx is NULL");
  SOS_CHECK_ARG(n_images >= 0 && height >= 0 && width >= 0 && n >= 0, "negative size");
  if (n == 0) return SOS_OK;
  SOS_CHECK_ARG(gray && kp_xy && desc, "NULL array");
  SOS_CHECK_ARG(n_images >= 1 && height > 2 * ORB_EDGE && width > 2 * ORB_EDGE, "image smaller than the ORB border");
  void* ws = nullptr;
  const int rc = sos_arena_get(ctx, sos_align_up((size_t)n_images * height * width, 256), &ws);
  if (rc != SOS_OK) return rc;
  return sos_orb_describe_into(ctx, gray, n_images, height, width, kp_xy, kp_angle_deg, kp_image, n, desc, keep, (uint8_t*)ws);
}

int sos_orb_describe_into(sos_ctx* ctx, const uint8_t* gray, int n_images, int height, int width, const float* kp_xy,
                          const float* kp_angle_deg, const int32_t* kp_image, int n, uint32_t* desc, uint8_t* keep,
                          uint8_t* blurred) {
  const int rc = sos_orb_blur(ctx, gray, n_images, height, width, blurred);
  if (rc != SOS_OK) return rc;
  orb_describe_kernel<<<sos_div_up(n, 8), 256, 0, ctx->stream>>>(blurred, height, width, (const float2*)kp_xy, kp_angle_deg,
                                                                 kp_image, n, desc, keep);
  SOS_LAUNCHED_AS(ctx, "orb_describe_kernel");
  return SOS_OK;
}
